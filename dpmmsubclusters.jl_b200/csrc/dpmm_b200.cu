// libdpmm_b200.so -- C ABI (include/dpmm_b200.h) over the sm_100a kernels of this directory.
// One context = one GPU = one shard of points = one "worker" of the reference
// (src/local_clusters_actions.jl *_worker! functions).  No CPU fallback exists: every entry point
// needs a CUDA device and reports DPMM_ECUDA otherwise.

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels_gauss.cuh"
#include "kernels_gauss_tc.cuh"
#include "kernels_gauss_tc2.cuh"
#include "kernels_ipc.cuh"
#include "kernels_mnm.cuh"
#include "kernels_mnm_tc.cuh"
#include "kernels_pack.cuh"
#include "kernels_params.cuh"
#include "kernels_params_mnm.cuh"
#include "kernels_sort.cuh"
#include "kernels_stats.cuh"
#include "kernels_stats_tc.cuh"
#include "kernels_stats_tc64.cuh"
#include "kernels_substats_tc.cuh"
#include "kernels_sublabel_tc64.cuh"

#include "ctx.cuh"
static int keff(const dpmm_ctx* c) { return std::max(std::max(c->K, c->label_bound), 1); }

static int nrec_floats(const dpmm_ctx* c) {
  if (c->prior == DPMM_PRIOR_MULTINOMIAL) return c->D;
  const int D = c->D;
  return gauss_col_off(D) + ((D + 3) & ~3);
}

// tables of the device-side parameter step: grown with their contents preserved
template <typename T>
static cudaError_t dev_grow_keep(T** p, size_t old_count, size_t new_count) {
  T* q = nullptr;
  cudaError_t e = cudaMalloc((void**)&q, std::max<size_t>(new_count, 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  e = cudaMemset(q, 0, std::max<size_t>(new_count, 1) * sizeof(T));
  if (e == cudaSuccess && *p && old_count) e = cudaMemcpy(q, *p, old_count * sizeof(T), cudaMemcpyDeviceToDevice);
  if (*p) cudaFree(*p);
  *p = q;
  return e;
}
// doubles per distribution of the posterior table
static int post_doubles(const dpmm_ctx* c) {
  return c->prior == DPMM_PRIOR_NIW ? NIW_POST_DOUBLES(c->D) : MNM_POST_DOUBLES(c->D);
}
static int ensure_tables(dpmm_ctx* ctx, int cap) {
  if (cap <= ctx->Kcap_tab) return 0;
  CK(cudaStreamSynchronize(ctx->stream));
  const int D = ctx->D, old = ctx->Kcap_tab;
  const bool niw = ctx->prior == DPMM_PRIOR_NIW;
  const size_t rec3 = (size_t)3 * (niw ? 1 + D + D * D : 1 + D), post3 = (size_t)3 * post_doubles(ctx);
  CK(dev_grow_keep(&ctx->ptab, old * rec3, cap * rec3));
  CK(dev_grow_keep(&ctx->ptab_alt, 0, cap * rec3));
  CK(dev_grow_keep(&ctx->post, old * post3, cap * post3));
  CK(dev_grow_keep(&ctx->post_alt, 0, cap * post3));
  if (niw) CK(dev_grow_keep(&ctx->lfac, (size_t)3 * old * D * D, (size_t)3 * cap * D * D));
  CK(dev_grow_keep(&ctx->pm_out, 0, (size_t)cap * 6 + (size_t)cap * cap + 2));
  CK(dev_grow_keep(&ctx->splittable_d, 0, (size_t)cap));
  CK(dev_grow_keep(&ctx->newof_d, 0, (size_t)cap));
  CK(dev_grow_keep(&ctx->w_out, (size_t)old, (size_t)cap));
  CK(dev_grow_keep(&ctx->lr_out, (size_t)2 * old, (size_t)2 * cap));
  ctx->Kcap_tab = cap;
  return 0;
}

static int ensure_k(dpmm_ctx* ctx, int K) {
  if (K <= ctx->Kcap) return 0;
  int cap = std::max(K, std::max(8, ctx->Kcap * 2));
  cap = std::min(cap, DPMM_MAX_K);
  if (K > cap) return fail(ctx, DPMM_ELIMIT, "K exceeds DPMM_MAX_K");
  // the stream may still read the old buffers
  CK(cudaStreamSynchronize(ctx->stream));
  const int D = ctx->D;
  ctx->rec_f = nrec_floats(ctx);
  ctx->stats_rec = (ctx->prior == DPMM_PRIOR_NIW) ? 1 + D + D * D : 1 + D;
  // preserve nothing: all K-sized buffers are rewritten by the next set_params / sort
  CK(dev_realloc(&ctx->recs, (size_t)3 * cap * ctx->rec_f));
  if (ctx->prior == DPMM_PRIOR_NIW) CK(dev_realloc(&ctx->raw_params, (size_t)3 * cap * (D + D * D + 1)));
  CK(dev_realloc(&ctx->cst, (size_t)3 * cap));
  CK(dev_realloc(&ctx->logw, (size_t)cap));
  CK(dev_realloc(&ctx->loglr, (size_t)2 * cap));
  if (ctx->prior == DPMM_PRIOR_MULTINOMIAL) CK(dev_realloc(&ctx->logp_t, (size_t)D * (cap + MNM_KT)));
  if (ctx->mtc_ok) {
    CK(dev_realloc(&ctx->mtc_w, (size_t)3 * ((D + 31) / 32) * MTC_N * 32));
    ctx->mtc_params = false;
  }
  if (ctx->tc_ok || ctx->t2_ok) {
    CK(dev_realloc(&ctx->tc_b, (size_t)cap * D));
    CK(dev_realloc(&ctx->tc_mu, (size_t)cap * D));
    CK(dev_realloc(&ctx->tc_fro, (size_t)cap));
    ctx->tc_params = ctx->t2_params = false;
  }
  if (ctx->t2_ok) {
    const int capt = std::min(cap, T2_MAX_K);   // beyond that the images do not fit shared memory anyway
    CK(dev_realloc(&ctx->t2_piv, (size_t)capt * D * D));
    CK(dev_realloc(&ctx->t2_u, (size_t)capt * D * D));
    CK(dev_realloc(&ctx->t2_scr, (size_t)gauss_tc2_nch(D, capt) * (D / 8) * 1024));
    CK(dev_realloc(&ctx->t2_bias, (size_t)capt * (gauss_tc2_nch(D, capt) * 512 + 32)));
    CK(dev_realloc(&ctx->t2_fro8, (size_t)capt));
  }
  if (ctx->tc_ok) {
    const int capc = std::min(cap, TC_MAX_K);
    CK(dev_realloc(&ctx->tc_w, (size_t)((capc + TC_NCL - 1) / TC_NCL) * TC_NCL * TC_D * TC_D));
    CK(dev_realloc(&ctx->ss_w, (size_t)cap * 2 * SS_D * SS_D));
    CK(dev_realloc(&ctx->ss_b, (size_t)cap * 2 * SS_D));
    CK(dev_realloc(&ctx->ss_c, (size_t)cap * SS_D));
    CK(dev_realloc(&ctx->lcount, (size_t)cap));
  }
  if (ctx->prior == DPMM_PRIOR_NIW && D == L64_D) {   // operands of the D = 64 tensor-core sub-label kernel
    CK(dev_realloc(&ctx->ss_w, (size_t)cap * 2 * D * D));
    CK(dev_realloc(&ctx->ss_b, (size_t)cap * 2 * D));
    CK(dev_realloc(&ctx->ss_c, (size_t)cap * D));
  }
  CK(dev_realloc(&ctx->hist_mem, (size_t)2 * cap));
  ctx->hist = ctx->hist_mem;
  ctx->hist_cur = ctx->hist_spare_clean = 0;
  ctx->t2_moved = nullptr;
  ctx->risk_zeroed_k = 0;
  CK(dev_realloc(&ctx->seg_off, (size_t)cap + 1));
  CK(dev_realloc(&ctx->scat_cursor, (size_t)cap));
  CK(dev_realloc(&ctx->lr_cursor, (size_t)2 * cap));
  CK(dev_realloc(&ctx->lut_l, (size_t)cap));
  CK(dev_realloc(&ctx->lut_r, (size_t)cap));
  CK(dev_realloc(&ctx->rule, (size_t)cap));
  CK(dev_realloc(&ctx->wanted, (size_t)cap));
  CK(dev_realloc(&ctx->idx_list, (size_t)cap));
  CK(dev_realloc(&ctx->acc, (size_t)2 * cap * ctx->stats_rec));
  CK(dev_realloc(&ctx->centers, (size_t)2 * cap * ctx->D));
  CK(dev_realloc(&ctx->outbuf, (size_t)3 * cap * ctx->stats_rec + 1));   // + the risk counter of the cached statistics
  ctx->items_cap = ctx->n / ctx->chunk + 2 * (int64_t)cap + 2;
  CK(dev_realloc(&ctx->items, (size_t)ctx->items_cap));
  ctx->Kcap = cap;
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  ctx->params_set = false;   // every parameter buffer above was reallocated: set_params must run again
  ctx->acc_cleared = ctx->cursors_fresh = false;
  if (ctx->dev_params) {
    int rc = ensure_tables(ctx, cap);
    if (rc) return rc;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// dispatch over the feature dimension (NIW): the kernels live in launch_niw.cu, one object per set
// ------------------------------------------------------------------------------------------------
#define DPMM_NIW_DIMS(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(12) X(16) X(24) X(32) X(48) X(64)

static bool niw_dim_supported(int D) {
  switch (D) {
#define X(d) case d:
    DPMM_NIW_DIMS(X)
#undef X
    return true;
    default:
      return false;
  }
}

#define DECL_SET(n)                                                                              \
  int niw_set_label_##n(dpmm_ctx*, const GaussLabelArgs&, int, int*);                            \
  int niw_set_sublabel_##n(dpmm_ctx*, const SubLabelArgs&, bool, int, int*);                     \
  int niw_set_stats_##n(dpmm_ctx*, const StatsArgs&, int, int*);
DECL_SET(0) DECL_SET(1) DECL_SET(2) DECL_SET(3) DECL_SET(4) DECL_SET(5)
#undef DECL_SET

int niw_launch_label(dpmm_ctx* ctx, const GaussLabelArgs& a) {
  int rc = DPMM_ELIMIT;
  const int D = ctx->D;
  if (niw_set_label_0(ctx, a, D, &rc) && niw_set_label_1(ctx, a, D, &rc) && niw_set_label_2(ctx, a, D, &rc) &&
      niw_set_label_3(ctx, a, D, &rc) && niw_set_label_4(ctx, a, D, &rc) && niw_set_label_5(ctx, a, D, &rc))
    return fail(ctx, DPMM_ELIMIT, "NIW: no kernel instantiated for this D");
  return rc;
}
int niw_launch_sublabel(dpmm_ctx* ctx, const SubLabelArgs& a, bool sample) {
  int rc = DPMM_ELIMIT;
  const int D = ctx->D;
  if (niw_set_sublabel_0(ctx, a, sample, D, &rc) && niw_set_sublabel_1(ctx, a, sample, D, &rc) &&
      niw_set_sublabel_2(ctx, a, sample, D, &rc) && niw_set_sublabel_3(ctx, a, sample, D, &rc) &&
      niw_set_sublabel_4(ctx, a, sample, D, &rc) && niw_set_sublabel_5(ctx, a, sample, D, &rc))
    return fail(ctx, DPMM_ELIMIT, "NIW: no kernel instantiated for this D");
  return rc;
}
int niw_launch_stats(dpmm_ctx* ctx, const StatsArgs& a) {
  int rc = DPMM_ELIMIT;
  const int D = ctx->D;
  if (niw_set_stats_0(ctx, a, D, &rc) && niw_set_stats_1(ctx, a, D, &rc) && niw_set_stats_2(ctx, a, D, &rc) &&
      niw_set_stats_3(ctx, a, D, &rc) && niw_set_stats_4(ctx, a, D, &rc) && niw_set_stats_5(ctx, a, D, &rc))
    return fail(ctx, DPMM_ELIMIT, "NIW: no kernel instantiated for this D");
  return rc;
}

// ------------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------------
extern "C" const char* dpmm_last_error(const dpmm_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

extern "C" int dpmm_limits(int32_t* out3) {
  if (!out3) return DPMM_EINVAL;
  out3[0] = 64;
  out3[1] = DPMM_MNM_MAX_D;
  out3[2] = DPMM_MAX_K;
  return 0;
}

extern "C" int dpmm_create(dpmm_ctx** out, const float* x, int64_t n_local, int32_t d, int32_t prior_kind,
                           int32_t device, uint64_t seed, int64_t global_offset) {
  dpmm_ctx* ctx = nullptr;
  if (!out) return fail(nullptr, DPMM_EINVAL, "out is NULL");
  *out = nullptr;
  NEED(x != nullptr && n_local > 0 && d > 0, DPMM_EINVAL, "x must be non-NULL with n_local > 0 and d > 0");
  NEED(n_local < ((int64_t)1 << 31) - 4096, DPMM_ELIMIT, "n_local must fit in int32 (shard the points over more GPUs)");
  NEED(prior_kind == DPMM_PRIOR_NIW || prior_kind == DPMM_PRIOR_MULTINOMIAL, DPMM_EINVAL, "unknown prior kind");
  int dpad = d;
  if (prior_kind == DPMM_PRIOR_NIW) {
    // kernels are instantiated for D in {1-8, 12, 16, 24, 32, 48, 64}; any other D <= 64 runs zero-padded to the
    // next width (padded features are 0 with mean 0 and unit precision: no likelihood or statistic changes, and the
    // D^2 constant keeps the caller's D)
    NEED(d <= 64, DPMM_ELIMIT, "NIW: D must be <= 64");
    while (!niw_dim_supported(dpad)) ++dpad;
  } else
    NEED(d <= DPMM_MNM_MAX_D, DPMM_ELIMIT, "multinomial: D must be <= 16384");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, DPMM_ECUDA, "no CUDA device: libdpmm_b200 has no CPU fallback");
  NEED(device >= 0 && device < ndev, DPMM_EINVAL, "bad device ordinal");
  ctx = new dpmm_ctx();
  ctx->device = device;
  ctx->n = n_local;
  ctx->D = dpad;
  ctx->D_user = d;
  ctx->prior = prior_kind;
  ctx->seed = seed;
  ctx->goff = global_offset;
  auto bail = [&](int code) {
    g_err = ctx->err;
    dpmm_destroy(ctx);
    return code;
  };
#define CKC(call)                                                                        \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                    \
      return bail(DPMM_ECUDA);                                                           \
    }                                                                                    \
  } while (0)
  CKC(cudaSetDevice(device));
  cudaDeviceProp prop;
  CKC(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    ctx->err = "device is not sm_100-class (Blackwell); this library ships sm_100a code only";
    return bail(DPMM_ECUDA);
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
  ctx->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  CKC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CKC(cudaMalloc((void**)&ctx->x, (size_t)n_local * dpad * sizeof(float)));
  CKC(cudaMalloc((void**)&ctx->labels, (size_t)n_local * sizeof(int32_t)));
  CKC(cudaMalloc((void**)&ctx->sub, (size_t)n_local));
  CKC(cudaMalloc((void**)&ctx->perm, (size_t)n_local * sizeof(int32_t)));
  CKC(cudaMalloc((void**)&ctx->perm2, (size_t)n_local * sizeof(int32_t)));
  CKC(cudaMalloc((void**)&ctx->item_ctr, 2 * sizeof(int32_t)));
  if (dpad == d) {
    CKC(cudaMemcpyAsync(ctx->x, x, (size_t)n_local * d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  } else {
    float* raw = nullptr;
    CKC(cudaMalloc((void**)&raw, (size_t)n_local * d * sizeof(float)));
    cudaError_t e1 = cudaMemcpyAsync(raw, x, (size_t)n_local * d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    if (e1 == cudaSuccess) {
      pad_points_kernel<<<(unsigned)prop.multiProcessorCount * 8, 256, 0, ctx->stream>>>(raw, n_local, d, dpad, ctx->x);
      e1 = cudaGetLastError();
    }
    if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(ctx->stream);
    cudaFree(raw);
    CKC(e1);
  }
  CKC(cudaMemsetAsync(ctx->labels, 0, (size_t)n_local * sizeof(int32_t), ctx->stream));
  CKC(cudaMemsetAsync(ctx->sub, 0, (size_t)n_local, ctx->stream));
  CKC(cudaStreamSynchronize(ctx->stream));
  if (prior_kind == DPMM_PRIOR_NIW && dpad == TC_D && n_local >= TC_TILE) {
    // TMA descriptor of X as a [n][32] float tensor, 128-point boxes, 128B swizzle (K2 operand A)
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn != nullptr &&
        qres == cudaDriverEntryPointSuccess) {
      const cuuint64_t gdim[2] = {(cuuint64_t)TC_D, (cuuint64_t)n_local};
      const cuuint64_t gstr[1] = {(cuuint64_t)TC_D * 4};
      const cuuint32_t box[2] = {TC_D, TC_TILE};
      const cuuint32_t estr[2] = {1, 1};
      const CUresult r = ((EncodeFn)fn)(&ctx->tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ctx->x, gdim, gstr, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      ctx->tc_ok = (r == CUDA_SUCCESS);
    }
  }
  if (ctx->tc_ok || (prior_kind == DPMM_PRIOR_NIW && (dpad == 32 || dpad == 64) && n_local >= T2_TILE)) {
    // two alternating counter sets [exact evaluations: points, evaluations | overflow count | pad]: the overflow
    // kernel of a call clears the set of the next one, so no memset launches sit between the sweeps
    CKC(cudaMalloc((void**)&ctx->ctr_sets, 2 * T2_CTR_SET * sizeof(int32_t)));
    CKC(cudaMemset(ctx->ctr_sets, 0, 2 * T2_CTR_SET * sizeof(int32_t)));
    ctx->tc_stats = ctx->ctr_sets;
    ctx->t2_ctr = ctx->ctr_sets + 2;
  }
  if (prior_kind == DPMM_PRIOR_NIW && (dpad == 32 || dpad == 64) && n_local >= T2_TILE) ctx->t2_ok = true;
  if (prior_kind == DPMM_PRIOR_MULTINOMIAL && d % 4 == 0 && d <= MTC_MAX_D && n_local >= MTC_TILE) {
    // the tensor-core likelihood is exact only for TF32-exact counts: integral, |x| < 2^11
    bool exact = false;
    {   // (on the device: the points are there already)
      int32_t* flag = nullptr;
      int32_t hflag = 1;
      if (cudaMalloc((void**)&flag, 4) == cudaSuccess) {
        cudaMemsetAsync(flag, 0, 4, ctx->stream);
        tf32_exact_scan_kernel<<<(unsigned)ctx->sm_count * 16, 256, 0, ctx->stream>>>(ctx->x, (int64_t)n_local * d, flag);
        if (cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
            cudaStreamSynchronize(ctx->stream) == cudaSuccess)
          exact = hflag == 0;
        cudaFree(flag);
      }
    }
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (exact && cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        fn != nullptr && qres == cudaDriverEntryPointSuccess) {
      const cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)n_local};
      const cuuint64_t gstr[1] = {(cuuint64_t)d * 4};
      const cuuint32_t box[2] = {32, MTC_TILE};
      const cuuint32_t estr[2] = {1, 1};
      const CUresult r = ((EncodeFn)fn)(&ctx->tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ctx->x, gdim, gstr, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      ctx->mtc_ok = (r == CUDA_SUCCESS);
    }
  }
#undef CKC
  // work-item length of the statistics kernels: NIW <= StatsCfg::MAX_CHUNK (a CTA per item);
  // multinomial items are taken by single warps, so they are shorter
  ctx->chunk = prior_kind == DPMM_PRIOR_NIW ? 1024 : 256;
  *out = ctx;
  return 0;
}

extern "C" int dpmm_destroy(dpmm_ctx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (env_int("DPMM_VERBOSE", 0))
    fprintf(stderr, "[dpmm] fused sub-label+statistics launches %lld, statistics served from them %lld, exact recomputations %lld\n",
            (long long)ctx->n_fused, (long long)ctx->n_cached, (long long)ctx->n_recompute);
  for (int p = 0; p < IPC_MAX_WORLD; ++p)
    if (ctx->ipc_peer[p]) cudaIpcCloseMemHandle(ctx->ipc_peer[p]);
  if (ctx->ipc_local) cudaFree(ctx->ipc_local);
  dpmm_internal_smart_free(ctx);
  if (ctx->side) {
    cudaStreamSynchronize(ctx->side);
    cudaStreamDestroy(ctx->side);
    cudaEventDestroy(ctx->ev_fork);
    cudaEventDestroy(ctx->ev_join);
  }
  if (ctx->comm && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(ctx->comm);
  for (auto& t : ctx->tev) {
    cudaEventDestroy(t.a);
    cudaEventDestroy(t.b);
  }
  for (auto e : ctx->ev_pool) cudaEventDestroy(e);
  void* ptrs[] = {ctx->x, ctx->labels, ctx->sub, ctx->perm, ctx->perm2, ctx->u_label, ctx->u_sub, ctx->r_bits,
                  ctx->raw_params, ctx->recs, ctx->cst, ctx->logw, ctx->loglr, ctx->logp_t, ctx->t2_piv, ctx->t2_scr, ctx->t2_u, ctx->t2_bias, ctx->t2_fro8, ctx->ctr_sets, ctx->tc_w, ctx->tc_b, ctx->tc_mu, ctx->tc_fro, ctx->ss_w, ctx->ss_b, ctx->ss_c, ctx->lcount, ctx->mtc_w, ctx->hist_mem, ctx->seg_off,
                  ctx->scat_cursor, ctx->lr_cursor, ctx->lut_l, ctx->lut_r, ctx->rule, ctx->wanted,
                  ctx->idx_list, ctx->acc, ctx->centers, ctx->outbuf, ctx->items, ctx->item_ctr, ctx->hyper_d, ctx->ptab,
                  ctx->ptab_alt, ctx->post, ctx->post_alt, ctx->lfac, ctx->pm_out, ctx->splittable_d, ctx->newof_d,
                  ctx->w_out, ctx->lr_out, ctx->wide, ctx->wide_status};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (ctx->hstage) cudaFreeHost(ctx->hstage);
  if (ctx->t2_hstat) cudaFreeHost(ctx->t2_hstat);
  if (ctx->t2_hstat_ev) cudaEventDestroy(ctx->t2_hstat_ev);
  for (int i = 0; i < 2; ++i) {
    if (ctx->hup[i]) cudaFreeHost(ctx->hup[i]);
    if (ctx->hup_ev[i]) cudaEventDestroy(ctx->hup_ev[i]);
  }
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return 0;
}

extern "C" int dpmm_set_stream(dpmm_ctx* ctx, void* cuda_stream) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return 0;
}

extern "C" int dpmm_sync(dpmm_ctx* ctx) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dpmm_set_sampler(dpmm_ctx* ctx, int32_t sampler) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(sampler == DPMM_SAMPLER_INVERSE_CDF || sampler == DPMM_SAMPLER_GUMBEL, DPMM_EINVAL, "unknown sampler");
  ctx->sampler = sampler;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// relabel plumbing
// ------------------------------------------------------------------------------------------------
static int run_relabel(dpmm_ctx* ctx, const std::vector<int32_t>& ll, const std::vector<int32_t>& lr,
                       const std::vector<uint8_t>& rule, bool uses_rng) {
  const int K = (int)ll.size();
  int rc = ensure_k(ctx, K);
  if (rc) return rc;
  const size_t b4 = (size_t)K * 4;
  void* hs = nullptr;
  const int slot = upload_acquire(ctx, 2 * b4 + K, &hs);
  if (slot < 0) return slot;
  char* h = (char*)hs;
  memcpy(h, ll.data(), b4);
  memcpy(h + b4, lr.data(), b4);
  memcpy(h + 2 * b4, rule.data(), K);
  CK(cudaMemcpyAsync(ctx->lut_l, h, b4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->lut_r, h + b4, b4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->rule, h + 2 * b4, K, cudaMemcpyHostToDevice, ctx->stream));
  rc = upload_release(ctx, slot);
  if (rc) return rc;
  if (uses_rng) ctx->call += 1;
  {
    KernelTimer kt(ctx, TK_RELABEL);
    const int T = 256;
    const unsigned grid = (unsigned)std::min<int64_t>((ctx->n + T - 1) / T, (int64_t)ctx->sm_count * 16);
    relabel_kernel<<<grid, T, 0, ctx->stream>>>(ctx->labels, ctx->sub, ctx->n, K, ctx->lut_l, ctx->lut_r, ctx->rule,
                                                ctx->r_bits, ctx->seed, ctx->call, ctx->goff);
    CK(cudaGetLastError());
  }
  return 0;
}

extern "C" int dpmm_init_labels(dpmm_ctx* ctx, int32_t init_clusters, int32_t outlier) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(init_clusters >= 1 && init_clusters + (outlier ? 1 : 0) <= DPMM_MAX_K, DPMM_EINVAL, "bad init_clusters");
  CK(cudaSetDevice(ctx->device));
  ctx->label_bound = init_clusters + (outlier ? 1 : 0);
  {
    int rc = ensure_k(ctx, ctx->label_bound);
    if (rc) return rc;
  }
  ctx->call += 1;
  {
    KernelTimer kt(ctx, TK_RELABEL);
    const int T = 256;
    const unsigned grid = (unsigned)std::min<int64_t>((ctx->n + T - 1) / T, (int64_t)ctx->sm_count * 16);
    init_labels_kernel<<<grid, T, 0, ctx->stream>>>(ctx->labels, ctx->n, init_clusters, outlier ? 1 : 0, ctx->seed,
                                                    ctx->call, ctx->goff);
    CK(cudaGetLastError());
  }
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  return dpmm_randomize_sublabels(ctx, nullptr, 0);
}

extern "C" int dpmm_randomize_sublabels(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  int K = keff(ctx);
  if (indices != nullptr) {
    for (int i = 0; i < n_indices; ++i) {
      NEED(indices[i] >= 1 && indices[i] <= DPMM_MAX_K, DPMM_EINVAL, "cluster index out of range");
      K = std::max<int>(K, (int)indices[i]);
    }
  }
  std::vector<int32_t> ll(K), lr(K);
  std::vector<uint8_t> rule(K, indices == nullptr ? 3 : 0);
  for (int k = 0; k < K; ++k) ll[k] = lr[k] = k;
  if (indices != nullptr) {
    if (n_indices == 0) return 0;
    for (int i = 0; i < n_indices; ++i) rule[indices[i] - 1] = 3;
  }
  ctx->partitioned = ctx->stats_cached = false;
  return run_relabel(ctx, ll, lr, rule, true);
}

extern "C" int dpmm_apply_split(dpmm_ctx* ctx, const int64_t* indices, const int64_t* new_indices, int32_t n) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  if (n == 0) return 0;
  NEED(indices && new_indices && n > 0, DPMM_EINVAL, "bad split lists");
  int K = keff(ctx);
  for (int i = 0; i < n; ++i) {
    NEED(indices[i] >= 1 && new_indices[i] >= 1 && indices[i] <= DPMM_MAX_K && new_indices[i] <= DPMM_MAX_K,
         DPMM_EINVAL, "cluster index out of range");
    K = std::max<int>(K, (int)std::max(indices[i], new_indices[i]));
  }
  // sequential semantics of the reference loop (local_clusters_actions.jl:269-277) composed into
  // one table: maps are tracked per ORIGINAL (label, side).
  std::vector<int32_t> ll(K), lr(K);
  std::vector<uint8_t> rule(K, 0);
  for (int k = 0; k < K; ++k) ll[k] = lr[k] = k;
  for (int i = 0; i < n; ++i) {
    const int idx = (int)indices[i] - 1, nw = (int)new_indices[i] - 1;
    for (int k = 0; k < K; ++k) {
      // points currently labelled idx: those whose left/right image is idx.  A point that already
      // received a fresh random sub-label (rule 3) has an unknown side; the reference only ever
      // issues disjoint splits, so reject the ambiguous case instead of guessing.
      const bool hit_l = ll[k] == idx, hit_r = lr[k] == idx;
      if (!hit_l && !hit_r) continue;
      NEED(rule[k] == 0 && hit_l && hit_r, DPMM_EINVAL, "split lists must be disjoint");
      lr[k] = nw;
      rule[k] = 3;
    }
  }
  ctx->label_bound = std::max(ctx->label_bound, K);
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  return run_relabel(ctx, ll, lr, rule, true);
}

extern "C" int dpmm_apply_merge(dpmm_ctx* ctx, const int64_t* indices, const int64_t* new_indices, int32_t n) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  if (n == 0) return 0;
  NEED(indices && new_indices && n > 0, DPMM_EINVAL, "bad merge lists");
  int K = keff(ctx);
  for (int i = 0; i < n; ++i) {
    NEED(indices[i] >= 1 && new_indices[i] >= 1 && indices[i] <= DPMM_MAX_K && new_indices[i] <= DPMM_MAX_K,
         DPMM_EINVAL, "cluster index out of range");
    K = std::max<int>(K, (int)std::max(indices[i], new_indices[i]));
  }
  // merge never looks at the sub-label, so the sequential loop (:297-303) composes exactly:
  // lab[k] = current label of points that started with label k, rule[k] = their forced side.
  std::vector<int32_t> lab(K);
  std::vector<uint8_t> rule(K, 0);
  for (int k = 0; k < K; ++k) lab[k] = k;
  for (int i = 0; i < n; ++i) {
    const int idx = (int)indices[i] - 1, nw = (int)new_indices[i] - 1;
    for (int k = 0; k < K; ++k)
      if (lab[k] == idx) rule[k] = 1;
    for (int k = 0; k < K; ++k)
      if (lab[k] == nw) {
        rule[k] = 2;
        lab[k] = idx;
      }
  }
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  return run_relabel(ctx, lab, lab, rule, false);
}

extern "C" int dpmm_remove_empty(dpmm_ctx* ctx, const int64_t* pts_count, int32_t k) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  NEED(pts_count && k >= 1 && k <= DPMM_MAX_K, DPMM_EINVAL, "bad pts_count");
  // remove_empty_clusters_worker! (:446-455): new = old - #{empty clusters with index < old}
  std::vector<int32_t> lab(k);
  std::vector<uint8_t> rule(k, 0);
  int removed = 0;
  bool any = false;
  for (int i = 0; i < k; ++i) {
    lab[i] = i - removed;
    if (pts_count[i] == 0) {
      ++removed;
      any = true;
    }
  }
  if (!any) return 0;
  NEED(ctx->label_bound <= k, DPMM_EINVAL, "pts_count is shorter than the number of label values in use");
  if (ctx->dev_params && ctx->Kcap_tab > 0) {
    // the persistent statistics / posterior tables follow the compaction
    const int kt_ = std::min(k, ctx->Kcap_tab);
    std::vector<int32_t> newof(kt_);
    for (int i = 0, r2 = 0; i < kt_; ++i) {
      newof[i] = pts_count[i] == 0 ? -1 : i - r2;
      if (pts_count[i] == 0) ++r2;
    }
    int rc2 = ensure_stage(ctx, (size_t)kt_ * 4);
    if (rc2) return rc2;
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->hstage, newof.data(), (size_t)kt_ * 4);
    CK(cudaMemcpyAsync(ctx->newof_d, ctx->hstage, (size_t)kt_ * 4, cudaMemcpyHostToDevice, ctx->stream));
    const int rec3 = 3 * ctx->stats_rec, post3 = 3 * post_doubles(ctx);
    KernelTimer kt(ctx, TK_PARAMS, 2);
    table_gather_kernel<<<dim3(8, (unsigned)kt_), 256, 0, ctx->stream>>>(ctx->ptab, ctx->newof_d, kt_, rec3, ctx->ptab_alt);
    table_gather_kernel<<<dim3(8, (unsigned)kt_), 256, 0, ctx->stream>>>(ctx->post, ctx->newof_d, kt_, post3, ctx->post_alt);
    CK(cudaGetLastError());
    std::swap(ctx->ptab, ctx->ptab_alt);
    std::swap(ctx->post, ctx->post_alt);
  }
  ctx->label_bound = std::max(1, k - removed);
  ctx->K = std::min(ctx->K, ctx->label_bound);  // parameters of the dropped clusters are stale anyway
  ctx->params_set = false;
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  return run_relabel(ctx, lab, lab, rule, false);
}

// ------------------------------------------------------------------------------------------------
// label gather / restore
// ------------------------------------------------------------------------------------------------
// scratch of n int64 on the device for the boundary conversions (allocated on first use)
static int ensure_wide(dpmm_ctx* ctx) {
  if (ctx->wide == nullptr) {
    CK(cudaMalloc((void**)&ctx->wide, (size_t)ctx->n * 8));
    CK(cudaMalloc((void**)&ctx->wide_status, 2 * sizeof(int32_t)));
  }
  return 0;
}
static unsigned stream_grid(const dpmm_ctx* ctx, int64_t n) {
  return (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 16);
}

extern "C" int dpmm_get_labels(dpmm_ctx* ctx, int64_t* out) {
  NEED(ctx && out, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_wide(ctx);
  if (rc) return rc;
  widen_labels_kernel<int32_t><<<stream_grid(ctx, ctx->n), 256, 0, ctx->stream>>>(ctx->labels, ctx->n, ctx->wide);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, ctx->wide, (size_t)ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dpmm_get_sublabels(dpmm_ctx* ctx, int64_t* out) {
  NEED(ctx && out, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_wide(ctx);
  if (rc) return rc;
  widen_labels_kernel<uint8_t><<<stream_grid(ctx, ctx->n), 256, 0, ctx->stream>>>(ctx->sub, ctx->n, ctx->wide);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, ctx->wide, (size_t)ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// upload `src` (n int64), narrow into dst on the device; returns the largest label in *mx; EINVAL on a bad value.
// The current labels are replaced only when every value is valid (narrowing goes through a scratch copy).
template <typename T>
static int set_labels_common(dpmm_ctx* ctx, const int64_t* src, int64_t hi, T* dst, int* mx, const char* what) {
  int rc = ensure_wide(ctx);
  if (rc) return rc;
  T* tmp = nullptr;
  CK(cudaMalloc((void**)&tmp, (size_t)ctx->n * sizeof(T)));
  cudaError_t e = cudaMemsetAsync(ctx->wide_status, 0, 8, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->wide, src, (size_t)ctx->n * 8, cudaMemcpyHostToDevice, ctx->stream);
  int32_t st[2] = {0, 1};
  if (e == cudaSuccess) {
    narrow_labels_kernel<T><<<stream_grid(ctx, ctx->n), 256, 0, ctx->stream>>>(ctx->wide, ctx->n, hi, tmp, ctx->wide_status);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(st, ctx->wide_status, 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess && st[1] == 0) e = cudaMemcpyAsync(dst, tmp, (size_t)ctx->n * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(tmp);
  if (e != cudaSuccess) return fail(ctx, DPMM_ECUDA, std::string("set labels: ") + cudaGetErrorString(e));
  if (st[1] != 0) return fail(ctx, DPMM_EINVAL, what);
  *mx = st[0];
  return 0;
}

extern "C" int dpmm_set_labels(dpmm_ctx* ctx, const int64_t* labels) {
  NEED(ctx && labels, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  int mx = 0;
  int rc = set_labels_common<int32_t>(ctx, labels, DPMM_MAX_K, ctx->labels, &mx, "label out of range [1, DPMM_MAX_K]");
  if (rc) return rc;
  ctx->label_bound = mx;
  rc = ensure_k(ctx, mx);
  if (rc) return rc;
  ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;
  return 0;
}

extern "C" int dpmm_set_sublabels(dpmm_ctx* ctx, const int64_t* sublabels) {
  NEED(ctx && sublabels, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  int mx = 0;
  int rc = set_labels_common<uint8_t>(ctx, sublabels, 2, ctx->sub, &mx, "sub-label must be 1 or 2");
  if (rc) return rc;
  ctx->partitioned = ctx->stats_cached = false;
  return 0;
}

extern "C" int dpmm_set_uniforms(dpmm_ctx* ctx, const double* u_label, const double* u_sub, const uint8_t* r_bits) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  auto put = [&](auto** dev, const auto* host, size_t bytes) -> cudaError_t {
    if (host == nullptr) {
      if (*dev) cudaFree(*dev);
      *dev = nullptr;
      return cudaSuccess;
    }
    if (*dev == nullptr) {
      cudaError_t e = cudaMalloc((void**)dev, bytes);
      if (e != cudaSuccess) return e;
    }
    return cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice);
  };
  CK(put(&ctx->u_label, u_label, (size_t)ctx->n * 8));
  CK(put(&ctx->u_sub, u_sub, (size_t)ctx->n * 8));
  CK(put(&ctx->r_bits, r_bits, (size_t)ctx->n));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------------
static void common_weights(dpmm_ctx* ctx, int K, const float* weights, const float* lr_weights, float* h_logw,
                           float* h_loglr) {
  // log(v) at local_clusters_actions.jl:126 and :92-93 is a Float32 log; evaluate in Float64 and
  // round once (matches the oracle's log_f32).
  for (int k = 0; k < K; ++k) h_logw[k] = (float)std::log((double)weights[k]);
  for (int k = 0; k < 2 * K; ++k) h_loglr[k] = (float)std::log((double)lr_weights[k]);
}

// Factor (unless `lfac` is given), pack and derive every parameter image of the sweep kernels from
// ctx->raw_params = [mu | invSigma | logdet] (device) for K clusters; logw / loglr are already in place.
static int niw_pack_launch(dpmm_ctx* ctx, int K, const double* lfac) {
  const int D = ctx->D, REC = ctx->rec_f, TRIP = gauss_col_off(D);
  const size_t nrec = (size_t)3 * K;
  const bool tcp = ctx->tc_ok && K <= TC_MAX_K;
  ctx->tc_params = ctx->t2_params = false;
  if (tcp) {
    const size_t wfl = (size_t)((K + TC_NCL - 1) / TC_NCL) * TC_NCL * TC_D * TC_D;
    CK(cudaMemsetAsync(ctx->tc_w, 0, wfl * 4, ctx->stream));   // zero padding of the last chunk
  }
  // second-generation label path: screen over all features while the images stay small, else over the last 8
  bool t2p = false;
  int t2_ks = 0, t2_nch = 0;
  if (ctx->t2_ok) {
    t2_nch = gauss_tc2_nch(D, K);
    t2_ks = (D == 32 && t2_nch <= 4) ? D : 8;
    t2p = K <= T2_MAX_K && GaussTc2Smem(D, K, t2_ks, t2_nch, std::max(K, ctx->label_bound) + 8).total <= (size_t)ctx->smem_optin;
    if (t2p) CK(cudaMemsetAsync(ctx->t2_scr, 0, (size_t)t2_nch * (t2_ks / 8) * 4096, ctx->stream));
  }
  {
    NiwPackArgs pa{};
    pa.D = D; pa.K = K; pa.rec_f = REC; pa.trip = TRIP; pa.D_const = ctx->D_user;
    pa.mu = ctx->raw_params; pa.inv_sigma = ctx->raw_params + nrec * D; pa.logdet = ctx->raw_params + nrec * D + nrec * D * D;
    pa.recs = ctx->recs; pa.cst = ctx->cst;
    pa.tc_w = tcp ? ctx->tc_w : nullptr; pa.tc_b = ctx->tc_b; pa.tc_mu = ctx->tc_mu; pa.tc_fro = ctx->tc_fro;
    pa.ss_w = (ctx->tc_ok || D == L64_D) ? ctx->ss_w : nullptr; pa.ss_b = ctx->ss_b; pa.ss_c = ctx->ss_c;
    pa.t2_piv = t2p ? ctx->t2_piv : nullptr; pa.t2_scr = ctx->t2_scr; pa.t2_u = ctx->t2_u; pa.t2_KS = t2_ks;
    pa.t2_n0 = gauss_tc2_n0(D); pa.t2_fro8 = ctx->t2_fro8; pa.lfac = lfac;
    KernelTimer kt(ctx, TK_PARAMS);
    niw_pack_kernel<<<(unsigned)nrec, NIW_PACK_THREADS, (size_t)D * (D + 1) * sizeof(double), ctx->stream>>>(pa);
    CK(cudaGetLastError());
  }
  if (t2p) {
    NiwT2BiasArgs ba{};
    ba.D = D; ba.K = K; ba.KS = t2_ks; ba.n0 = gauss_tc2_n0(D); ba.nch = t2_nch; ba.u = ctx->t2_u; ba.mu = ctx->tc_mu;
    ba.bias = ctx->t2_bias;
    KernelTimer kt(ctx, TK_PARAMS);
    niw_t2_bias_kernel<<<(unsigned)K, 256, 0, ctx->stream>>>(ba);
    CK(cudaGetLastError());
  }
  ctx->tc_params = tcp;
  ctx->t2_params = t2p;
  ctx->t2_KS = t2_ks;
  ctx->t2_nch = t2_nch;
  ctx->K = K;
  ctx->params_set = true;
  return 0;
}

extern "C" int dpmm_set_params_niw(dpmm_ctx* ctx, int32_t K, const float* mu, const float* inv_sigma,
                                   const float* logdet, const float* weights, const float* lr_weights) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(ctx->prior == DPMM_PRIOR_NIW, DPMM_ESTATE, "context was created with the multinomial prior");
  NEED(K >= 1 && K <= DPMM_MAX_K, DPMM_ELIMIT, "K out of range");
  NEED(mu && inv_sigma && logdet && weights && lr_weights, DPMM_EINVAL, "NULL parameter array");
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_k(ctx, K);
  if (rc) return rc;
  const int D = ctx->D, Du = ctx->D_user;
  const size_t nrec = (size_t)3 * K;
  // raw parameters -> pinned staging -> device; the factorisation and packing run on the device
  const size_t raw_floats = nrec * D + nrec * D * D + nrec;
  const size_t bytes = (raw_floats + K + 2 * K) * sizeof(float);
  void* hs = nullptr;
  const int slot = upload_acquire(ctx, bytes, &hs);   // alternating pinned buffers: no stream synchronisation
  if (slot < 0) return slot;
  float* h_mu = (float*)hs;
  float* h_inv = h_mu + nrec * D;
  float* h_ld = h_inv + nrec * D * D;
  float* h_logw = h_ld + nrec;
  float* h_loglr = h_logw + K;
  if (Du == D) {
    memcpy(h_mu, mu, nrec * D * 4);
    memcpy(h_inv, inv_sigma, nrec * D * D * 4);
  } else {   // padded features: mean 0, unit precision, uncorrelated with the rest
    memset(h_mu, 0, nrec * D * 4);
    memset(h_inv, 0, nrec * D * D * 4);
    for (size_t t = 0; t < nrec; ++t) {
      memcpy(h_mu + t * D, mu + t * Du, (size_t)Du * 4);
      for (int i = 0; i < Du; ++i) memcpy(h_inv + (t * D + i) * D, inv_sigma + (t * Du + i) * Du, (size_t)Du * 4);
      for (int i = Du; i < D; ++i) h_inv[(t * D + i) * D + i] = 1.f;
    }
  }
  memcpy(h_ld, logdet, nrec * 4);
  common_weights(ctx, K, weights, lr_weights, h_logw, h_loglr);
  CK(cudaMemcpyAsync(ctx->raw_params, h_mu, raw_floats * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->logw, h_logw, (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->loglr, h_loglr, (size_t)2 * K * 4, cudaMemcpyHostToDevice, ctx->stream));
  rc = upload_release(ctx, slot);
  if (rc) return rc;
  rc = niw_pack_launch(ctx, K, nullptr);
  if (rc) return rc;
  return 0;
}

// Derive the sweep kernels' images from the [3K][D] log-probabilities in ctx->recs (the transposed table and, on the
// tensor-core path, the TF32 split); logw / loglr are already in place.
static int mnm_pack_launch(dpmm_ctx* ctx, int K) {
  const int D = ctx->D;
  const int KP = (K + MNM_KT - 1) / MNM_KT * MNM_KT;
  const bool mtc = ctx->mtc_ok && K <= MTC_MAX_K;
  MnmPackArgs pa{};
  pa.D = D; pa.K = K; pa.KP = KP; pa.logp = ctx->recs; pa.logp_t = ctx->logp_t; pa.mtc_w = mtc ? ctx->mtc_w : nullptr;
  const int64_t ne = std::max<int64_t>((int64_t)D * KP, mtc ? (int64_t)((D + 31) / 32) * MTC_N * 32 : 0);
  {
    KernelTimer kt(ctx, TK_PARAMS);
    mnm_pack_kernel<<<(unsigned)std::min<int64_t>((ne + 255) / 256, (int64_t)ctx->sm_count * 4), 256, 0, ctx->stream>>>(pa);
    CK(cudaGetLastError());
  }
  ctx->mtc_params = mtc;
  ctx->K = K;
  ctx->KP = KP;
  ctx->params_set = true;
  return 0;
}

extern "C" int dpmm_set_params_multinomial(dpmm_ctx* ctx, int32_t K, const float* log_p, const float* weights,
                                           const float* lr_weights) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(ctx->prior == DPMM_PRIOR_MULTINOMIAL, DPMM_ESTATE, "context was created with the NIW prior");
  NEED(K >= 1 && K <= DPMM_MAX_K, DPMM_ELIMIT, "K out of range");
  NEED(log_p && weights && lr_weights, DPMM_EINVAL, "NULL parameter array");
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_k(ctx, K);
  if (rc) return rc;
  const int D = ctx->D;
  const size_t nrec = (size_t)3 * K;
  const size_t bytes = (nrec * D + K + 2 * K) * sizeof(float);
  void* hs = nullptr;
  const int slot = upload_acquire(ctx, bytes, &hs);
  if (slot < 0) return slot;
  float* h_recs = (float*)hs;
  float* h_logw = h_recs + nrec * D;
  float* h_loglr = h_logw + K;
  memcpy(h_recs, log_p, nrec * D * 4);
  common_weights(ctx, K, weights, lr_weights, h_logw, h_loglr);
  CK(cudaMemcpyAsync(ctx->recs, h_recs, nrec * D * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->logw, h_logw, (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->loglr, h_loglr, (size_t)2 * K * 4, cudaMemcpyHostToDevice, ctx->stream));
  rc = upload_release(ctx, slot);
  if (rc) return rc;
  return mnm_pack_launch(ctx, K);
}

// ------------------------------------------------------------------------------------------------
// the sweep
// ------------------------------------------------------------------------------------------------
static int ensure_sorted(dpmm_ctx* ctx);

// The sweep's kernels are chained with programmatic dependent launch (common.cuh).  The label and fused kernels allocate
// tensor memory before their grid dependency, i.e. possibly while CTAs of the previous kernel still run.  That is safe
// when no two CTAs that hold tensor memory can share an SM, which their register footprints decide (C2: 448 x 128 and
// 896 x 72 registers of 64 Ki): checked here once from the compiled kernels; if it does not hold, these two kernels are
// launched without the attribute.  Timed launches (KernelTimer events between the kernels) are plain as well.
static bool sweep_pdl_ok(dpmm_ctx* ctx) {
  if (ctx->pdl_tmem < 0) {
    const struct { const void* f; int threads; } ks[] = {{(const void*)gauss_label_tc2_kernel<32>, T2_THREADS(32)},
                                                        {(const void*)gauss_label_tc2_kernel<64>, T2_THREADS(64)},
                                                        {(const void*)niw_substats_tc_kernel, SS_THREADS}};
    int regs_sm = 0;
    bool ok = cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, ctx->device) == cudaSuccess;
    int foot[3];
    for (int i = 0; i < 3 && ok; ++i) {
      cudaFuncAttributes fa;
      ok = cudaFuncGetAttributes(&fa, ks[i].f) == cudaSuccess;
      foot[i] = fa.numRegs * ks[i].threads;
    }
    for (int i = 0; i < 3 && ok; ++i)
      for (int j = 0; j < 3; ++j) ok &= foot[i] + foot[j] > regs_sm;
    cudaGetLastError();
    ctx->pdl_tmem = ok ? 1 : 0;
  }
  return ctx->pdl_tmem == 1 && !ctx->timing;
}

template <int D>
static int launch_label_tc2(dpmm_ctx* ctx, int final_iter, int nkeys) {
  const int K = ctx->K;
  GaussTc2Args a{};
  a.x = ctx->x; a.n = ctx->n; a.K = K; a.KS = ctx->t2_KS; a.nch = ctx->t2_nch; a.n0 = gauss_tc2_n0(D);
  a.perm = ctx->perm; a.seg_off = ctx->seg_off; a.nkeys = nkeys; a.wpiv = ctx->t2_piv; a.wscr = ctx->t2_scr;
  a.wbias = ctx->t2_bias; a.fro8 = ctx->t2_fro8;
  a.urows = ctx->t2_u; a.mu = ctx->tc_mu; a.cst = ctx->cst; a.logw = ctx->logw; a.fro = ctx->tc_fro;
  // this call's counter set (the other one was cleared by the previous call's overflow kernel)
  ctx->ctr_cur ^= 1;
  ctx->tc_stats = ctx->ctr_sets + T2_CTR_SET * ctx->ctr_cur;
  ctx->t2_ctr = ctx->tc_stats + 2;
  a.labels = ctx->labels; a.hist = ctx->hist; a.ovf_list = ctx->perm2; a.ovf_count = ctx->t2_ctr;
  a.u_inj = ctx->u_label; a.seed = ctx->seed; a.call = ctx->call; a.goff = ctx->goff; a.final_iter = final_iter;
  a.stats = ctx->tc_stats;
  a.moved = ctx->tc_stats + 4;
  const size_t sm = GaussTc2Smem(D, K, a.KS, a.nch, nkeys).total;
  CK(cudaFuncSetAttribute(gauss_label_tc2_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  if (!ctx->ctr_clean) CK(cudaMemsetAsync(ctx->ctr_sets, 0, 2 * T2_CTR_SET * sizeof(int32_t), ctx->stream));   // another path used them
  if (ctx->t2_hstat == nullptr) {
    CK(cudaHostAlloc((void**)&ctx->t2_hstat, 4 * sizeof(int32_t), cudaHostAllocMapped));
    CK(cudaHostGetDevicePointer((void**)&ctx->t2_hstat_dev, ctx->t2_hstat, 0));
    CK(cudaEventCreateWithFlags(&ctx->t2_hstat_ev, cudaEventDisableTiming));
  }
  const int64_t grid = std::min<int64_t>((ctx->n + T2_TILE - 1) / T2_TILE, (int64_t)ctx->sm_count);
  {
    KernelTimer kt(ctx, TK_LABEL);
    CK(launch_pdl(sweep_pdl_ok(ctx), gauss_label_tc2_kernel<D>, (unsigned)grid, T2_THREADS(D), sm, ctx->stream, a));
  }
  // the (normally empty) overflow list: points with a NaN / Inf screen value or more than 7 candidates
  GaussListArgs l{};
  l.x = ctx->x; l.K = K; l.list = ctx->perm2; l.count = ctx->t2_ctr; l.urows = ctx->t2_u; l.mu = ctx->tc_mu;
  l.cst = ctx->cst; l.logw = ctx->logw; l.labels = ctx->labels; l.hist = ctx->hist; l.u_inj = ctx->u_label;
  l.seed = ctx->seed; l.call = ctx->call; l.goff = ctx->goff; l.final_iter = final_iter; l.stats = a.stats;
  l.moved = a.moved;
  l.zero_next = ctx->ctr_sets + T2_CTR_SET * (ctx->ctr_cur ^ 1);
  ctx->ctr_clean = true;
  // the histogram buffer of the previous labels is not read again: it becomes the next call's, cleared here
  l.zero_hist = ctx->hist_mem + (size_t)(ctx->hist_cur ^ 1) * ctx->Kcap;
  l.zero_hist_n = K;
  ctx->hist_spare_clean = K;
  // the counters go to mapped host memory; the event behind the kernel says they have arrived (never waited for)
  l.hstat = ctx->t2_hstat_dev;
  // the last block of the overflow kernel scans the new label histogram (label_scan_kernel's job) when the scan's
  // width is the K of this call: one launch fewer between the label kernel and the sort
  l.ticket = ctx->tc_stats + 3; l.scan_k = K; l.seg_off = ctx->seg_off; l.scat_cursor = ctx->scat_cursor; l.lr_cursor = ctx->lr_cursor;
  const size_t lsm = (size_t)8 * K * 4;
  if (lsm > 48 * 1024) CK(cudaFuncSetAttribute(gauss_label_list_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm));
  {
    KernelTimer kt(ctx, TK_LABEL_OVF);
    CK(launch_pdl(!ctx->timing, gauss_label_list_kernel<D>, (unsigned)ctx->sm_count * 2, 256, lsm, ctx->stream, l));
  }
  CK(cudaEventRecord(ctx->t2_hstat_ev, ctx->stream));
  ctx->t2_hstat_pending = true;
  return 0;
}

template <int TP>
static int launch_mnm_label_stream(dpmm_ctx* ctx, MnmLabelArgs& a) {
  const size_t sm = MnmStreamCfg<TP>::smem_bytes(a.K);
  NEED(sm <= (size_t)ctx->smem_optin, DPMM_ELIMIT, "internal: multinomial streaming label kernel does not fit shared memory");
  a.ntiles = (a.n + TP - 1) / TP;
  CK(cudaFuncSetAttribute(mnm_label_stream_kernel<TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mnm_label_stream_kernel<TP>, 256, sm));
  occ = std::max(occ, 1);
  const int64_t grid = std::min<int64_t>(a.ntiles, (int64_t)ctx->sm_count * occ);
  KernelTimer kt(ctx, TK_LABEL);
  mnm_label_stream_kernel<TP><<<(unsigned)grid, 256, sm, ctx->stream>>>(a);
  CK(cudaGetLastError());
  return 0;
}

static int run_sample_labels(dpmm_ctx* ctx, int final_iter, float* dump) {
  NEED(ctx->params_set, DPMM_ESTATE, "set_params must precede sample_labels");
  const int K = ctx->K;
  ctx->call += 1;
  // K2 second generation (tcgen05, D = 32 / 64, any K that fits): walks the points in the order of the
  // CURRENT label sort, so that sort has to be valid (it is, from the previous iteration, unless a relabel
  // operation ran since)
  bool use_t2 = ctx->prior == DPMM_PRIOR_NIW && ctx->t2_params && dump == nullptr &&
                ctx->sampler == DPMM_SAMPLER_INVERSE_CDF && env_int("DPMM_LABEL_TC", 2) == 2;
  if (use_t2 && env_int("DPMM_LABEL_ADAPT", 1) != 0) {
    // the previous tensor-core call's counters, if they have arrived: exact (point, cluster) evaluations cost about
    // what the FMA kernel pays per (point, cluster) too, so beyond ~K/3 of them per point (or many overflow points,
    // which evaluate all K) the FMA kernel that evaluates everything wins; try the tensor-core path again later
    if (ctx->t2_hstat_pending && cudaEventQuery(ctx->t2_hstat_ev) == cudaSuccess) {
      ctx->t2_hstat_pending = false;
      const double pts = std::max(1, ctx->t2_hstat[0]);
      const double evals = (double)ctx->t2_hstat[1] / pts;   // (overflow points count K evaluations each)
      if (evals > 0.03 * K + 0.05) ctx->t2_cooldown = 8;
    }
    if (ctx->t2_cooldown > 0) {
      --ctx->t2_cooldown;
      use_t2 = false;
    }
  }
  int nkeys = 0;
  if (use_t2) {
    nkeys = keff(ctx);
    use_t2 = GaussTc2Smem(ctx->D, K, ctx->t2_KS, ctx->t2_nch, nkeys).total <= (size_t)ctx->smem_optin;
  }
  if (use_t2) {
    int rc = ensure_sorted(ctx);
    if (rc) return rc;
  }
  if (use_t2 && ctx->hist_spare_clean >= K) {   // cleared by the previous tensor-core call's overflow kernel
    ctx->hist_cur ^= 1;
    ctx->hist = ctx->hist_mem + (size_t)ctx->hist_cur * ctx->Kcap;
    ctx->hist_spare_clean = 0;
  } else {
    CK(cudaMemsetAsync(ctx->hist, 0, (size_t)K * 4, ctx->stream));
  }
  if (use_t2) {
    int rc = ctx->D == 32 ? launch_label_tc2<32>(ctx, final_iter, nkeys) : launch_label_tc2<64>(ctx, final_iter, nkeys);
    if (rc) return rc;
  } else if (ctx->prior == DPMM_PRIOR_NIW && ctx->tc_params && dump == nullptr && ctx->sampler == DPMM_SAMPLER_INVERSE_CDF &&
      env_int("DPMM_LABEL_TC", 2) != 0) {
    // K2: tcgen05 TF32 screen + FP32 refine
    GaussTcArgs a{};
    a.n = ctx->n; a.K = K; a.wmat = ctx->tc_w; a.bvec = ctx->tc_b; a.mu = ctx->tc_mu; a.cst = ctx->cst; a.logw = ctx->logw;
    a.fro = ctx->tc_fro; a.labels = ctx->labels; a.hist = ctx->hist; a.u_inj = ctx->u_label; a.seed = ctx->seed;
    a.call = ctx->call; a.goff = ctx->goff; a.final_iter = final_iter; a.ntiles = (ctx->n + TC_TILE - 1) / TC_TILE;
    a.stats = env_int("DPMM_TC_STATS", 0) ? ctx->tc_stats : nullptr;
    const size_t sm = GaussTcSmem(K).total;
    NEED(sm <= (size_t)ctx->smem_optin, DPMM_ELIMIT, "internal: tensor-core label kernel does not fit shared memory");
    CK(cudaFuncSetAttribute(gauss_label_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    const int64_t grid = std::min<int64_t>((a.ntiles + 1) / 2, (int64_t)ctx->sm_count);
    if (a.stats) {
      CK(cudaMemsetAsync(ctx->tc_stats, 0, 8, ctx->stream));
      ctx->ctr_clean = false;
    }
    KernelTimer kt(ctx, TK_LABEL);
    gauss_label_tc_kernel<<<(unsigned)grid, TC_THREADS, sm, ctx->stream>>>(ctx->tmap_x, a);
    CK(cudaGetLastError());
  } else if (ctx->prior == DPMM_PRIOR_NIW) {
    GaussLabelArgs a{};
    a.x = ctx->x; a.n = ctx->n; a.K = K; a.recs = ctx->recs; a.cst = ctx->cst; a.logw = ctx->logw;
    a.labels = ctx->labels; a.hist = ctx->hist; a.u_inj = ctx->u_label; a.seed = ctx->seed; a.call = ctx->call;
    a.goff = ctx->goff; a.final_iter = final_iter; a.sampler = ctx->sampler; a.dump = dump;
    int rc = niw_launch_label(ctx, a);
    if (rc) return rc;
  } else if (ctx->mtc_params && dump == nullptr && env_int("DPMM_LABEL_TC", 1) != 0) {
    // K3 on tcgen05: exact TF32 3-way split GEMM of counts x log-probabilities
    MnmTcArgs a{};
    a.n = ctx->n; a.D = ctx->D; a.K = K; a.NP = (ctx->D + 31) / 32; a.wsplit = ctx->mtc_w; a.logw = ctx->logw;
    a.labels = ctx->labels; a.hist = ctx->hist; a.u_inj = ctx->u_label; a.seed = ctx->seed; a.call = ctx->call;
    a.goff = ctx->goff; a.final_iter = final_iter; a.sampler = ctx->sampler; a.ntiles = (ctx->n + MTC_TILE - 1) / MTC_TILE;
    a.NG = MnmTcSmem(K, a.NP, MTC_NG).total <= (size_t)ctx->smem_optin ? MTC_NG : 2;
    const size_t sm = MnmTcSmem(K, a.NP, a.NG).total;
    NEED(sm <= (size_t)ctx->smem_optin, DPMM_ELIMIT, "internal: multinomial tensor-core kernel does not fit shared memory");
    CK(cudaFuncSetAttribute(mnm_label_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    const int64_t grid = std::min<int64_t>(a.ntiles, (int64_t)ctx->sm_count);
    KernelTimer kt(ctx, TK_LABEL);
    mnm_label_tc_kernel<<<(unsigned)grid, MTC_THREADS(a.NG), sm, ctx->stream>>>(ctx->tmap_x, a);
    CK(cudaGetLastError());
  } else {
    MnmLabelArgs a{};
    a.x = ctx->x; a.n = ctx->n; a.D = ctx->D; a.DS = ctx->D | 1; a.K = K; a.KP = ctx->KP; a.logp_t = ctx->logp_t;
    a.logw = ctx->logw; a.labels = ctx->labels; a.hist = ctx->hist; a.u_inj = ctx->u_label; a.seed = ctx->seed;
    a.call = ctx->call; a.goff = ctx->goff; a.final_iter = final_iter; a.sampler = ctx->sampler; a.dump = dump;
    int T = 128;
    auto bytes = [&](int T_) { return ((size_t)a.D * a.KP + (size_t)T_ * a.DS + (size_t)K * T_) * 4 + (size_t)K * 4; };
    while (T > 32 && bytes(T) > (size_t)ctx->smem_optin) T /= 2;
    if (bytes(T) <= (size_t)ctx->smem_optin) {
      a.ntiles = (a.n + T - 1) / T;
      const size_t sm = bytes(T);
      CK(cudaFuncSetAttribute(mnm_label_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      int occ = 1;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mnm_label_kernel, T, sm));
      occ = std::max(occ, 1);
      const int64_t grid = std::min<int64_t>(a.ntiles, (int64_t)ctx->sm_count * occ);
      KernelTimer kt(ctx, TK_LABEL);
      mnm_label_kernel<<<(unsigned)grid, T, sm, ctx->stream>>>(a);
      CK(cudaGetLastError());
    } else {
      // the table does not fit shared memory: stream it in feature panels (largest point tile whose parr slice fits)
      int rc = MnmStreamCfg<128>::smem_bytes(K) <= (size_t)ctx->smem_optin ? launch_mnm_label_stream<128>(ctx, a)
             : MnmStreamCfg<64>::smem_bytes(K) <= (size_t)ctx->smem_optin  ? launch_mnm_label_stream<64>(ctx, a)
                                                                            : launch_mnm_label_stream<32>(ctx, a);
      if (rc) return rc;
    }
  }
  ctx->hist_valid = true;
  ctx->scan_valid = use_t2;   // the overflow kernel's last block already scanned the new histogram (width K)
  ctx->t2_moved = use_t2 ? ctx->tc_stats + 4 : nullptr;   // (perm sorts the labels this call started from)
  ctx->sorted = false;
  ctx->partitioned = ctx->stats_cached = false;
  ctx->label_bound = K;
  return 0;
}

static int ensure_sorted(dpmm_ctx* ctx) {
  if (ctx->sorted) return 0;
  const int K = keff(ctx);
  {
    int rc = ensure_k(ctx, K);
    if (rc) return rc;
  }
  KernelTimer kt(ctx, TK_SORT, 1 + (ctx->hist_valid ? 0 : 1) + (ctx->hist_valid && ctx->scan_valid ? 0 : 1));
  if (!ctx->hist_valid) {
    CK(cudaMemsetAsync(ctx->hist, 0, (size_t)K * 4, ctx->stream));
    const int T = 256;
    const unsigned grid = (unsigned)std::min<int64_t>((ctx->n + T - 1) / T, (int64_t)ctx->sm_count * 8);
    label_hist_kernel<<<grid, T, (size_t)K * 4, ctx->stream>>>(ctx->labels, ctx->n, K, ctx->hist);
    CK(cudaGetLastError());
    ctx->hist_valid = true;
  }
  if (!(ctx->hist_valid && ctx->scan_valid)) {
    label_scan_kernel<<<1, 1024, 0, ctx->stream>>>(ctx->hist, K, ctx->seg_off, ctx->scat_cursor, ctx->lr_cursor);
    CK(cudaGetLastError());
  }
  // the tensor-core label call that produced these labels counted the points that changed label: with none, perm
  // (sorted for the labels that call started from) is still a valid sort and the scatter kernel skips its work
  const int32_t* moved = ctx->hist_valid && ctx->scan_valid ? ctx->t2_moved : nullptr;
  ctx->t2_moved = nullptr;
  ctx->scan_valid = false;   // the scatter below consumes the cursors
  {
    const int T = 256;
    const unsigned grid = (unsigned)((ctx->n + (int64_t)T * SCATTER_PPT - 1) / ((int64_t)T * SCATTER_PPT));
    // the fused sub-label + statistics kernel (NIW, D = 32) wants its accumulators cleared, and the statistics finalise
    // that follows it the risk slot of outbuf: done here
    const bool pre = ctx->prior == DPMM_PRIOR_NIW && ctx->D == SS_D && ctx->tc_ok && ctx->lcount != nullptr;
    CK(launch_pdl(!ctx->timing, label_scatter_kernel, grid, T, (size_t)K * 8, ctx->stream, (const int32_t*)ctx->labels,
                  ctx->n, K, ctx->scat_cursor, ctx->perm, pre ? ctx->acc : nullptr, pre ? (int64_t)2 * K * ctx->stats_rec : (int64_t)0,
                  pre ? ctx->lcount : nullptr, pre ? K : 0, pre ? ctx->outbuf + (size_t)K * 3 * ctx->stats_rec : nullptr, moved));
    ctx->acc_cleared = pre;
    ctx->risk_zeroed_k = pre ? K : 0;
  }
  ctx->sorted = true;
  ctx->partitioned = ctx->stats_cached = false;
  ctx->cursors_fresh = true;
  return 0;
}

int dpmm_internal_ensure_sorted(dpmm_ctx* ctx) { return ensure_sorted(ctx); }

// sub-label draw (sample=true) or partition only (sample=false); both leave perm2 partitioned.
static int run_sublabels(dpmm_ctx* ctx, bool sample, float* dump) {
  int rc = ensure_sorted(ctx);
  if (rc) return rc;
  if (!ctx->cursors_fresh) {
    // cursors were consumed by a previous partition of the same sort: rebuild them
    KernelTimer kt(ctx, TK_SORT);
    label_scan_kernel<<<1, 1024, 0, ctx->stream>>>(ctx->hist, keff(ctx), ctx->seg_off, ctx->scat_cursor,
                                                   ctx->lr_cursor);
    CK(cudaGetLastError());
  }
  SubLabelArgs a{};
  a.x = ctx->x; a.n = ctx->n; a.K = ctx->K; a.recs = ctx->recs; a.cst = ctx->cst; a.loglr = ctx->loglr;
  a.labels = ctx->labels; a.sub = ctx->sub; a.perm = ctx->perm; a.perm2 = ctx->perm2; a.cursor = ctx->lr_cursor;
  a.seg_off = ctx->seg_off;
  a.u_inj = ctx->u_sub; a.seed = ctx->seed; a.call = ctx->call; a.goff = ctx->goff; a.dump = dump; a.D = ctx->D;
  // K4+K5 fused on tcgen05 (NIW, D = 32): the sub-label draw also accumulates the left / right statistics
  // of every cluster, which the next dpmm_suff_stats calls serve from the accumulators.
  if (sample && ctx->prior == DPMM_PRIOR_NIW && ctx->D == SS_D && ctx->tc_ok && env_int("DPMM_SUBSTATS_TC", 1) != 0 &&
      SubStatsSmem(ctx->K).total <= (size_t)ctx->smem_optin && keff(ctx) == ctx->K) {
    const int K = ctx->K, recs = ctx->stats_rec;
    if (!ctx->acc_cleared) {   // (cleared by the label scatter kernel when the sort has just run)
      CK(cudaMemsetAsync(ctx->acc, 0, (size_t)2 * K * recs * 8, ctx->stream));
      CK(cudaMemsetAsync(ctx->lcount, 0, (size_t)K * 4, ctx->stream));
    }
    ctx->acc_cleared = false;
    SubStatsArgs f{};
    f.x = ctx->x; f.n = ctx->n; f.K = K; f.perm = ctx->perm; f.seg_off = ctx->seg_off; f.w = ctx->ss_w; f.bias = ctx->ss_b;
    f.cen = ctx->ss_c; f.cst = ctx->cst; f.loglr = ctx->loglr; f.sub = ctx->sub; f.acc = ctx->acc; f.rec = recs;
    f.lcount = ctx->lcount; f.centers = ctx->centers; f.u_inj = ctx->u_sub; f.seed = ctx->seed; f.call = ctx->call;
    f.goff = ctx->goff; f.dump = dump;
    const size_t smem = SubStatsSmem(K).total;
    CK(cudaFuncSetAttribute(niw_substats_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    {
      KernelTimer kt(ctx, TK_SUBLABEL);
      CK(launch_pdl(sweep_pdl_ok(ctx), niw_substats_tc_kernel, (unsigned)ctx->sm_count, SS_THREADS, smem, ctx->stream, f));
    }
    ctx->partitioned = false;
    ctx->stats_cached = true;
    ++ctx->n_fused;
    return 0;
  }
  // D = 64 on tcgen05: the draw and the left / right partition of perm2
  if (sample && ctx->prior == DPMM_PRIOR_NIW && ctx->D == L64_D && ctx->ss_w != nullptr && env_int("DPMM_SUBLABEL_TC64", 1) != 0 &&
      SubLabel64Smem(ctx->K).total <= (size_t)ctx->smem_optin && keff(ctx) == ctx->K && ctx->n >= L64_TILE) {
    SubLabel64Args f{};
    f.x = ctx->x; f.n = ctx->n; f.K = ctx->K; f.perm = ctx->perm; f.seg_off = ctx->seg_off; f.w = ctx->ss_w; f.bias = ctx->ss_b;
    f.cen = ctx->ss_c; f.cst = ctx->cst; f.loglr = ctx->loglr; f.sub = ctx->sub; f.u_inj = ctx->u_sub; f.seed = ctx->seed;
    f.call = ctx->call; f.goff = ctx->goff; f.dump = dump; f.perm2 = ctx->perm2; f.cursor = ctx->lr_cursor;
    const size_t smem = SubLabel64Smem(ctx->K).total;
    CK(cudaFuncSetAttribute(niw_sublabel_tc64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    KernelTimer kt(ctx, TK_SUBLABEL);
    niw_sublabel_tc64_kernel<<<ctx->sm_count, L64_THREADS, smem, ctx->stream>>>(f);
    CK(cudaGetLastError());
    ctx->partitioned = true;       // the kernel's epilogue partitioned perm2 (and consumed the cursors)
    ctx->cursors_fresh = false;
    ctx->stats_cached = false;
    return 0;
  }
  if (ctx->prior == DPMM_PRIOR_NIW) {
    rc = niw_launch_sublabel(ctx, a, sample);
    if (rc) return rc;
  } else {
    const int T = 128;
    const unsigned grid = (unsigned)((a.n + T - 1) / T);
    KernelTimer kt(ctx, TK_SUBLABEL);
    if (sample && ctx->D <= 128)
      mnm_sublabel2_kernel<<<grid, T, 0, ctx->stream>>>(a);
    else if (sample && ctx->D > 1024)
      mnm_sublabel_staged_kernel<<<grid, MNM_SLS_T, 0, ctx->stream>>>(a);
    else if (sample)
      mnm_sublabel_kernel<true><<<grid, T, 0, ctx->stream>>>(a);
    else
      mnm_sublabel_kernel<false><<<grid, T, 0, ctx->stream>>>(a);
    CK(cudaGetLastError());
  }
  ctx->partitioned = true;
  ctx->cursors_fresh = false;
  return 0;
}

extern "C" int dpmm_sample_labels(dpmm_ctx* ctx, int32_t final_iter) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  return run_sample_labels(ctx, final_iter, nullptr);
}

extern "C" int dpmm_sample_sublabels(dpmm_ctx* ctx) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  NEED(ctx->params_set, DPMM_ESTATE, "set_params must precede sample_sublabels");
  NEED(ctx->label_bound <= ctx->K, DPMM_ESTATE, "labels refer to clusters beyond the K of set_params");
  ctx->call += 1;
  return run_sublabels(ctx, true, nullptr);
}

// The device part of a statistics call: accumulate, finalise into ctx->outbuf ([m][3][rec] (+ the risk counter of
// the fused path)) and all-reduce.  m = 0 when the index list is empty.
struct StatsCall {
  int m = 0;
  bool all = false, cached = false;
};
static int stats_compute(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices, StatsCall* sc) {
  const int K = keff(ctx);
  int rc = ensure_k(ctx, K);
  if (rc) return rc;
  const int D = ctx->D, rec = ctx->stats_rec;
  std::vector<int32_t> idx;
  if (indices == nullptr) {
    idx.resize(K);
    for (int k = 0; k < K; ++k) idx[k] = k;
  } else {
    NEED(n_indices >= 0, DPMM_EINVAL, "n_indices < 0");
    idx.resize(n_indices);
    for (int i = 0; i < n_indices; ++i) {
      NEED(indices[i] >= 1 && indices[i] <= K, DPMM_EINVAL, "cluster index out of range [1, K]");
      idx[i] = (int32_t)indices[i] - 1;
    }
  }
  const int m = (int)idx.size();
  sc->m = m;
  if (m == 0) return 0;
  NEED(m <= ctx->Kcap, DPMM_EINVAL, "more indices than clusters");
  const bool cached = ctx->stats_cached;   // accumulators of every cluster left by the fused sub-label kernel
  if (!cached && !ctx->partitioned) {
    rc = run_sublabels(ctx, false, nullptr);
    if (rc) return rc;
  }
  const bool all = (indices == nullptr);
  sc->all = all;
  sc->cached = cached;
  rc = ensure_stage(ctx, std::max<size_t>((size_t)m * 4 + K, ((size_t)m * 3 * rec + 1) * 8));
  if (rc) return rc;
  if (!all) {   // "all" needs no index list (the finalise kernel then uses k = a) and hence no host round trip here
    CK(cudaStreamSynchronize(ctx->stream));   // staging buffer reuse
    int32_t* h_idx = (int32_t*)ctx->hstage;
    uint8_t* h_w = (uint8_t*)(h_idx + m);
    memcpy(h_idx, idx.data(), (size_t)m * 4);
    CK(cudaMemcpyAsync(ctx->idx_list, h_idx, (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
    memset(h_w, 0, K);
    for (int v : idx) h_w[v] = 1;
    CK(cudaMemcpyAsync(ctx->wanted, h_w, K, cudaMemcpyHostToDevice, ctx->stream));
  }
  // K5 on tcgen05: all clusters of a D = 32 NIW model (no work list: CTAs own ranges of the tile sequence)
  const bool stats_tc = !cached && ctx->prior == DPMM_PRIOR_NIW && D == STC_D && all && ctx->tc_ok &&
                        env_int("DPMM_STATS_TC", 1) != 0 && StatsTcSmem(K).total <= (size_t)ctx->smem_optin;
  // ... and of a D = 64 model (kernels_stats_tc64.cuh)
  const bool stats_tc64 = !cached && ctx->prior == DPMM_PRIOR_NIW && D == S64_D && all && env_int("DPMM_STATS_TC", 1) != 0 &&
                          StatsTc64Smem(K).total <= (size_t)ctx->smem_optin;
  if (cached) {
    // nothing to accumulate
  } else if (!stats_tc && !stats_tc64) {
    KernelTimer kt(ctx, TK_STATS_AUX);
    stats_worklist_kernel<<<1, 256, (size_t)2 * K * 4, ctx->stream>>>(ctx->seg_off, ctx->lr_cursor,
                                                                      all ? nullptr : ctx->wanted, K, ctx->chunk,
                                                                      ctx->items, ctx->item_ctr, ctx->item_ctr + 1);
    CK(cudaGetLastError());
  }
  if (!cached) {
    CK(cudaMemsetAsync(ctx->acc, 0, (size_t)2 * K * rec * 8, ctx->stream));
    ctx->acc_cleared = false;   // about to be written by the separate statistics kernels
  }
  StatsArgs sa{};
  sa.x = ctx->x; sa.D = D; sa.perm2 = ctx->perm2; sa.items = ctx->items; sa.n_items = ctx->item_ctr;
  sa.next_item = ctx->item_ctr + 1; sa.acc = ctx->acc; sa.rec = rec;
  if (cached) {
    // served from the accumulators
  } else if (stats_tc) {
    StatsTcArgs ta{};
    ta.x = ctx->x; ta.perm2 = ctx->perm2; ta.seg_off = ctx->seg_off; ta.lr_cursor = ctx->lr_cursor; ta.K = K;
    ta.acc = ctx->acc; ta.rec = rec; ta.centers = ctx->centers;
    {
      KernelTimer kt(ctx, TK_STATS_AUX);
      stats_centers_kernel<<<2 * K, 256, 0, ctx->stream>>>(ctx->x, ctx->perm2, ctx->seg_off, ctx->lr_cursor, ctx->centers);
      CK(cudaGetLastError());
    }
    const size_t smem = StatsTcSmem(K).total;
    CK(cudaFuncSetAttribute(niw_stats_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(niw_stats_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // two CTAs per SM when their shared memory fits (every CTA owns a contiguous slice of the tile
    // sequence, so the grid size is free)
    const int occ = 2 * (smem + 1024) <= (size_t)ctx->smem_per_sm ? 2 : 1;
    KernelTimer kt(ctx, TK_STATS);
    niw_stats_tc_kernel<<<ctx->sm_count * occ, STC_THREADS, smem, ctx->stream>>>(ta);
    CK(cudaGetLastError());
  } else if (stats_tc64) {
    StatsTcArgs ta{};
    ta.x = ctx->x; ta.perm2 = ctx->perm2; ta.seg_off = ctx->seg_off; ta.lr_cursor = ctx->lr_cursor; ta.K = K;
    ta.acc = ctx->acc; ta.rec = rec; ta.centers = ctx->centers;
    {
      KernelTimer kt(ctx, TK_STATS_AUX);
      stats_centers64_kernel<<<2 * K, 512, 0, ctx->stream>>>(ctx->x, ctx->perm2, ctx->seg_off, ctx->lr_cursor, ctx->centers);
      CK(cudaGetLastError());
    }
    const size_t smem = StatsTc64Smem(K).total;
    CK(cudaFuncSetAttribute(niw_stats_tc64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    KernelTimer kt(ctx, TK_STATS);
    niw_stats_tc64_kernel<<<ctx->sm_count, S64_THREADS, smem, ctx->stream>>>(ta);
    CK(cudaGetLastError());
  } else if (ctx->prior == DPMM_PRIOR_NIW) {
    rc = niw_launch_stats(ctx, sa);
    if (rc) return rc;
  } else {
    const auto kern = D > 32 * MNM_STATS_NREG ? mnm_stats_kernel<true> : mnm_stats_kernel<false>;
    int occ = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, 0));
    occ = std::max(occ, 1);
    KernelTimer kt(ctx, TK_STATS);
    kern<<<ctx->sm_count * occ, 256, 0, ctx->stream>>>(sa);
    CK(cudaGetLastError());
  }
  // with a communicator and mapped peer memory the packed statistics go straight into this rank's exchange
  // buffer and one kernel reduces over NVLink; otherwise they go to outbuf (and through ncclAllReduce)
  const size_t nred = (size_t)m * 3 * rec + 1;
  const bool use_ipc = ctx->comm != nullptr && ctx->ipc_ok && nred <= ctx->ipc_cap;
  const uint32_t epoch = use_ipc ? ++ctx->ipc_epoch : 0;
  double* fin = use_ipc ? reinterpret_cast<double*>(ctx->ipc_local + IPC_FLAG_BYTES) + (size_t)(epoch & 1) * ctx->ipc_cap : ctx->outbuf;
  {
    KernelTimer kt(ctx, TK_STATS_AUX);
    const int T = 256;
    dim3 grid((unsigned)std::min((rec + T - 1) / T, 64), (unsigned)m);
    // the risk slot: cleared by the label scatter that preceded the fused kernel, or here
    if (!(fin == ctx->outbuf && m == ctx->risk_zeroed_k)) CK(cudaMemsetAsync(fin + (size_t)m * 3 * rec, 0, 8, ctx->stream));
    ctx->risk_zeroed_k = 0;
    CK(launch_pdl(!ctx->timing, stats_finalize_kernel, grid, T, 0, ctx->stream, (const double*)ctx->acc, (const int32_t*)ctx->seg_off,
                  (const int32_t*)ctx->lr_cursor, (const int32_t*)(all ? nullptr : ctx->idx_list), m, D, rec,
                  ctx->prior == DPMM_PRIOR_NIW ? 1 : 0, fin, (const float*)((stats_tc || stats_tc64 || cached) ? ctx->centers : nullptr),
                  (const int32_t*)(cached ? ctx->lcount : nullptr), cached ? fin + (size_t)m * 3 * rec : nullptr));
  }
  if (use_ipc) {
    IpcReduceArgs ia{};
    ia.world = ctx->world; ia.rank = ctx->rank; ia.epoch = epoch; ia.n = nred; ia.out = ctx->outbuf;
    ia.my_flags = reinterpret_cast<const uint32_t*>(ctx->ipc_local);
    for (int r = 0; r < ctx->world; ++r) {
      uint8_t* base = r == ctx->rank ? ctx->ipc_local : ctx->ipc_peer[r];
      ia.src[r] = reinterpret_cast<const double*>(base + IPC_FLAG_BYTES) + (size_t)(epoch & 1) * ctx->ipc_cap;
      ia.peer_flags[r] = reinterpret_cast<uint32_t*>(base);
    }
    KernelTimer kt(ctx, TK_ALLREDUCE);
    const unsigned grid = (unsigned)std::min<size_t>((nred / 2 + 255) / 256, (size_t)ctx->sm_count * 4);
    ipc_allreduce_kernel<<<grid, 256, 0, ctx->stream>>>(ia);
    CK(cudaGetLastError());
  } else if (ctx->comm != nullptr) {
    KernelTimer kt(ctx, TK_ALLREDUCE);
    // aggregate_suff_stats across workers (niw.jl:64-66; local_clusters_actions.jl:194-196, 246-248)
    // (the risk slot always travels, so the element count cannot differ between ranks)
    const int r = ctx->nccl.AllReduce(ctx->outbuf, ctx->outbuf, (size_t)m * 3 * rec + 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0,
                                      ctx->comm, ctx->stream);
    if (r != 0) return fail(ctx, DPMM_ENCCL, std::string("ncclAllReduce: ") + ctx->nccl.GetErrorString(r));
  }
  return 0;
}

extern "C" int dpmm_suff_stats(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices, int64_t* counts,
                               double* sum_x, double* sum_xx) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  if (indices == nullptr && n_indices > 0)
    NEED(n_indices == keff(ctx), DPMM_EINVAL,
         "indices == NULL means every cluster: n_indices must be 0 or the number of label values in use "
         "(max of the K of set_params and the largest label); the output arrays hold that many rows");
  StatsCall sc;
  int rc = stats_compute(ctx, indices, n_indices, &sc);
  if (rc) return rc;
  const int m = sc.m, D = ctx->D, rec = ctx->stats_rec;
  const bool cached = sc.cached;
  if (m == 0) return 0;
  if (counts == nullptr && sum_x == nullptr && sum_xx == nullptr) return 0;
  double* h = (double*)ctx->hstage;
  CK(cudaMemcpyAsync(h, ctx->outbuf, ((size_t)m * 3 * rec + (cached ? 1 : 0)) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (cached && h[(size_t)m * 3 * rec] != 0.0) {
    // some (tiny or degenerate) run lies far from its cluster's centre relative to its own magnitude:
    // recompute with the FP32/FP64 statistics kernel (on every rank: the counter was all-reduced)
    ctx->stats_cached = false;
    ++ctx->n_recompute;
    return dpmm_suff_stats(ctx, indices, n_indices, counts, sum_x, sum_xx);
  }
  if (cached) ++ctx->n_cached;
  for (int a = 0; a < m; ++a)
    for (int s = 0; s < 3; ++s) {
      const double* r = h + ((size_t)a * 3 + s) * rec;
      if (counts) counts[a * 3 + s] = (int64_t)llround(r[0]);
      const int Du = ctx->D_user;
      if (sum_x) memcpy(sum_x + ((size_t)a * 3 + s) * Du, r + 1, (size_t)Du * 8);
      if (sum_xx && ctx->prior == DPMM_PRIOR_NIW)
        for (int i = 0; i < Du; ++i)
          memcpy(sum_xx + (((size_t)a * 3 + s) * Du + i) * Du, r + 1 + D + (size_t)i * D, (size_t)Du * 8);
    }
  return 0;
}


// ------------------------------------------------------------------------------------------------
// device-side parameter step (NIW and multinomial): SURVEY.md 8f-1
// ------------------------------------------------------------------------------------------------
extern "C" int dpmm_num_clusters(const dpmm_ctx* ctx) { return ctx ? keff(ctx) : 0; }

extern "C" int dpmm_set_hyper_niw(dpmm_ctx* ctx, double kappa, const double* m, double nu, const double* psi, double alpha) {
  NEED(ctx && m && psi, DPMM_EINVAL, "NULL argument");
  NEED(ctx->prior == DPMM_PRIOR_NIW, DPMM_ESTATE, "context was created with the multinomial prior");
  NEED(ctx->D == ctx->D_user, DPMM_ELIMIT,
       "the device-side parameter step needs an instantiated feature dimension (1-8, 12, 16, 24, 32, 48, 64); "
       "sample the parameters on the host (dpmm_set_params_niw) for other D");
  NEED(kappa > 0 && nu > ctx->D - 1 && alpha > 0, DPMM_EINVAL, "need kappa > 0, nu > D - 1, alpha > 0");
  CK(cudaSetDevice(ctx->device));
  const int D = ctx->D;
  std::vector<double> h(NIW_HYPER_DOUBLES(D));
  // logdet psi by a host Cholesky of the symmetrised matrix (one-time, D <= 64)
  std::vector<double> A((size_t)D * D);
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) A[(size_t)i * D + j] = 0.5 * (psi[(size_t)i * D + j] + psi[(size_t)j * D + i]);
  double logdet = 0.0;
  for (int j = 0; j < D; ++j) {
    double d = A[(size_t)j * D + j];
    for (int k = 0; k < j; ++k) d -= A[(size_t)j * D + k] * A[(size_t)j * D + k];
    NEED(d > 0 && std::isfinite(d), DPMM_EINVAL, "psi must be positive definite");
    const double l = std::sqrt(d);
    A[(size_t)j * D + j] = l;
    logdet += 2.0 * std::log(l);
    for (int i = j + 1; i < D; ++i) {
      double v = A[(size_t)i * D + j];
      for (int k = 0; k < j; ++k) v -= A[(size_t)i * D + k] * A[(size_t)j * D + k];
      A[(size_t)i * D + j] = v / l;
    }
  }
  // niw_hyperparams stores kappa and nu as Float32 (niw.jl:6-11)
  const double kf = (double)(float)kappa, nf = (double)(float)nu;
  float lmv = (float)((double)D * (D - 1) / 4.0 * 1.1447298858494002);
  for (int j = 1; j <= D; ++j) lmv = (float)((double)lmv + std::lgamma(nf / 2.0 + (1.0 - j) / 2.0));
  h[0] = kf; h[1] = nf; h[2] = logdet; h[3] = (double)lmv;
  for (int i = 0; i < D; ++i) h[4 + i] = m[i];
  for (int e = 0; e < D * D; ++e) h[4 + D + e] = psi[e];
  if (!ctx->hyper_d) CK(cudaMalloc((void**)&ctx->hyper_d, h.size() * 8));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(ctx->hyper_d, h.data(), h.size() * 8, cudaMemcpyHostToDevice));
  ctx->alpha = (double)(float)alpha;   // model_hyper_params.alpha is Float32 (ds.jl:9)
  ctx->dev_params = true;
  return ensure_tables(ctx, std::max(ctx->Kcap, 8));
}

extern "C" int dpmm_set_hyper_multinomial(dpmm_ctx* ctx, const float* alpha_prior, double alpha) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(ctx->prior == DPMM_PRIOR_MULTINOMIAL, DPMM_ESTATE, "context was created with the NIW prior");
  NEED(alpha_prior, DPMM_EINVAL, "alpha_prior is NULL");
  NEED(alpha > 0, DPMM_EINVAL, "need alpha > 0");
  CK(cudaSetDevice(ctx->device));
  const int D = ctx->D;
  std::vector<double> h(MNM_HYPER_DOUBLES(D));
  double sa = 0.0;
  for (int d = 0; d < D; ++d) {
    NEED(std::isfinite(alpha_prior[d]) && alpha_prior[d] > 0.f, DPMM_EINVAL, "every alpha_prior[d] must be finite and > 0");
    h[2 + d] = (double)alpha_prior[d];
    sa += h[2 + d];
  }
  h[0] = sa;
  h[1] = std::lgamma(sa);
  if (!ctx->hyper_d) CK(cudaMalloc((void**)&ctx->hyper_d, h.size() * 8));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(ctx->hyper_d, h.data(), h.size() * 8, cudaMemcpyHostToDevice));
  ctx->alpha = (double)(float)alpha;
  ctx->dev_params = true;
  return ensure_tables(ctx, std::max(ctx->Kcap, 8));
}

#define DPMM_NEED_HYPER(what) \
  NEED(ctx->dev_params, DPMM_ESTATE, "dpmm_set_hyper_niw or dpmm_set_hyper_multinomial must precede " what)

static size_t niw_post_smem(int D) { return ((size_t)D * (D + 1) + 2 * D) * sizeof(double); }

// posterior + log marginal likelihood of the listed clusters (device list idx_d, or all m = K in order) from the table
static int launch_post(dpmm_ctx* ctx, const int32_t* idx_d, int m, double* out) {
  if (ctx->prior == DPMM_PRIOR_MULTINOMIAL) {
    MnmPostArgs pa{};
    pa.D = ctx->D; pa.rec = ctx->stats_rec; pa.hyper = ctx->hyper_d; pa.ptab = ctx->ptab; pa.idx_list = idx_d;
    pa.post = ctx->post; pa.out = out;
    KernelTimer kt(ctx, TK_PARAMS);
    mnm_post_kernel<<<dim3((unsigned)m, 3), MNM_PARAM_THREADS, 0, ctx->stream>>>(pa);
    CK(cudaGetLastError());
    return 0;
  }
  NiwPostArgs pa{};
  pa.D = ctx->D; pa.rec = ctx->stats_rec; pa.hyper = ctx->hyper_d; pa.ptab = ctx->ptab; pa.idx_list = idx_d;
  pa.post = ctx->post; pa.out = out;
  const size_t sm = niw_post_smem(ctx->D);
  if (sm > 48 * 1024) CK(cudaFuncSetAttribute(niw_post_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  KernelTimer kt(ctx, TK_PARAMS);
  niw_post_kernel<<<dim3((unsigned)m, 3), 256, sm, ctx->stream>>>(pa);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int dpmm_posterior_step(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices, int32_t from_table,
                                   const uint8_t* splittable, int32_t k_merge, int64_t* counts, double* logml,
                                   double* merge_logml) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  DPMM_NEED_HYPER("dpmm_posterior_step");
  const int rec = ctx->stats_rec;
  int m = 0;
  bool all = indices == nullptr;
  bool cached = false;
  if (!from_table) {
    StatsCall sc;
    int rc = stats_compute(ctx, indices, n_indices, &sc);
    if (rc) return rc;
    m = sc.m;
    cached = sc.cached;
    if (m == 0) return 0;
    rc = ensure_tables(ctx, ctx->Kcap);
    if (rc) return rc;
    const int rec3 = 3 * rec;
    dim3 grid((unsigned)std::min((rec3 + 255) / 256, 32), (unsigned)m);
    KernelTimer kt(ctx, TK_PARAMS);
    ptab_scatter_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->outbuf, all ? nullptr : ctx->idx_list, m, rec3, ctx->ptab);
    CK(cudaGetLastError());
  } else {
    // re-evaluate table rows (after dpmm_params_merge): the index list goes up by itself
    NEED(indices != nullptr && n_indices >= 0, DPMM_EINVAL, "from_table needs an index list");
    m = n_indices;
    if (m == 0) return 0;
    NEED(m <= ctx->Kcap_tab, DPMM_EINVAL, "more indices than clusters");
    int rc = ensure_stage(ctx, (size_t)m * 4);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    int32_t* h_idx = (int32_t*)ctx->hstage;
    for (int i = 0; i < m; ++i) {
      NEED(indices[i] >= 1 && indices[i] <= ctx->Kcap_tab, DPMM_EINVAL, "cluster index out of range");
      h_idx[i] = (int32_t)indices[i] - 1;
    }
    CK(cudaMemcpyAsync(ctx->idx_list, h_idx, (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
    all = false;
  }
  // the K x K table of merged log marginal likelihoods reads the statistics table only: it runs on the side stream
  // next to the posteriors
  const bool want_merge = merge_logml != nullptr && splittable != nullptr && k_merge > 1;
  double* merge_d = ctx->pm_out + (size_t)m * 6;
  if (want_merge) {
    NEED(k_merge <= ctx->Kcap_tab, DPMM_EINVAL, "k_merge exceeds the number of clusters");
    CK(cudaMemcpyAsync(ctx->splittable_d, splittable, (size_t)k_merge, cudaMemcpyHostToDevice, ctx->stream));
    const dim3 grid((unsigned)k_merge, (unsigned)k_merge);
    if (ctx->prior == DPMM_PRIOR_MULTINOMIAL) {
      MnmMergeArgs ma{};
      ma.D = ctx->D; ma.rec = rec; ma.K = k_merge; ma.hyper = ctx->hyper_d; ma.ptab = ctx->ptab;
      ma.splittable = ctx->splittable_d; ma.out = merge_d;
      int rcf = side_fork(ctx);
      if (rcf) return rcf;
      ctx->launches += 1;
      mnm_merge_kernel<<<grid, MNM_PARAM_THREADS, 0, ctx->side>>>(ma);
    } else {
      NiwMergeArgs ma{};
      ma.D = ctx->D; ma.rec = rec; ma.K = k_merge; ma.hyper = ctx->hyper_d; ma.ptab = ctx->ptab;
      ma.splittable = ctx->splittable_d; ma.out = merge_d;
      const size_t sm = niw_post_smem(ctx->D);
      if (sm > 48 * 1024) CK(cudaFuncSetAttribute(niw_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      int rcf = side_fork(ctx);
      if (rcf) return rcf;
      ctx->launches += 1;
      niw_merge_kernel<<<grid, 256, sm, ctx->side>>>(ma);
    }
    CK(cudaGetLastError());
  }
  int rc = launch_post(ctx, all ? nullptr : ctx->idx_list, m, ctx->pm_out);
  if (rc) return rc;
  if (want_merge) {
    rc = side_join(ctx);
    if (rc) return rc;
  }
  if (counts == nullptr && logml == nullptr && !want_merge) return 0;
  const size_t nd = (size_t)m * 6 + (want_merge ? (size_t)k_merge * k_merge : 0);
  rc = ensure_stage(ctx, (nd + 1) * 8);
  if (rc) return rc;
  double* h = (double*)ctx->hstage;
  CK(cudaMemcpyAsync(h, ctx->pm_out, nd * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (cached) CK(cudaMemcpyAsync(h + nd, ctx->outbuf + (size_t)m * 3 * rec, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (cached && h[nd] != 0.0) {
    // the fused accumulators were rejected (see dpmm_suff_stats): recompute exactly, on every rank
    ctx->stats_cached = false;
    ++ctx->n_recompute;
    return dpmm_posterior_step(ctx, indices, n_indices, from_table, splittable, k_merge, counts, logml, merge_logml);
  }
  if (cached) ++ctx->n_cached;
  for (int a = 0; a < m * 3; ++a) {
    if (counts) counts[a] = (int64_t)llround(h[2 * a]);
    if (logml) logml[a] = h[2 * a + 1];
  }
  if (want_merge) memcpy(merge_logml, h + (size_t)m * 6, (size_t)k_merge * k_merge * 8);
  return 0;
}

extern "C" int dpmm_sample_params(dpmm_ctx* ctx, int32_t K, int32_t from_prior, int32_t unit_weights) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  DPMM_NEED_HYPER("dpmm_sample_params");
  NEED(K >= 1 && K <= DPMM_MAX_K, DPMM_ELIMIT, "K out of range");
  int rc = ensure_k(ctx, K);
  if (rc) return rc;
  rc = ensure_tables(ctx, ctx->Kcap);
  if (rc) return rc;
  const int D = ctx->D;
  const size_t nrec = (size_t)3 * K;
  ctx->pcall += 1;
  {   // the Dirichlet weights depend on the posterior table only: side stream, next to the draws and the packing
    WeightsArgs wa{};
    wa.K = K; wa.D = D; wa.post = ctx->post; wa.stride = post_doubles(ctx); wa.alpha = ctx->alpha; wa.logw = ctx->logw;
    wa.loglr = ctx->loglr; wa.w_out = ctx->w_out; wa.lr_out = ctx->lr_out; wa.seed = ctx->seed; wa.call = ctx->pcall;
    wa.unit = unit_weights;
    rc = side_fork(ctx);
    if (rc) return rc;
    ctx->launches += 1;
    dpmm_weights_kernel<<<1, 256, (size_t)(K + 1) * 8, ctx->side>>>(wa);
    CK(cudaGetLastError());
  }
  if (ctx->prior == DPMM_PRIOR_MULTINOMIAL) {
    MnmDrawArgs da{};
    da.D = D; da.hyper = ctx->hyper_d; da.post = ctx->post; da.logp = ctx->recs; da.seed = ctx->seed; da.call = ctx->pcall;
    da.first = from_prior;
    {
      KernelTimer kt(ctx, TK_PARAMS);
      const size_t sm = (size_t)D * sizeof(double);
      if (sm > 48 * 1024) CK(cudaFuncSetAttribute(mnm_draw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      mnm_draw_kernel<<<(unsigned)nrec, MNM_PARAM_THREADS, sm, ctx->stream>>>(da);
      CK(cudaGetLastError());
    }
    rc = mnm_pack_launch(ctx, K);
    if (rc) return rc;
    return side_join(ctx);
  }
  {
    NiwDrawArgs da{};
    da.D = D; da.mu = ctx->raw_params; da.logdet = ctx->raw_params + nrec * D + nrec * D * D; da.hyper = ctx->hyper_d;
    da.post = ctx->post; da.lfac = ctx->lfac; da.seed = ctx->seed; da.call = ctx->pcall; da.first = from_prior;
    const size_t sm = ((size_t)3 * D * (D + 1) + 2 * D) * sizeof(double);
    if (sm > 48 * 1024) CK(cudaFuncSetAttribute(niw_draw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    KernelTimer kt(ctx, TK_PARAMS);
    niw_draw_kernel<<<(unsigned)nrec, NIW_PACK_THREADS, sm, ctx->stream>>>(da);
    CK(cudaGetLastError());
  }
  rc = niw_pack_launch(ctx, K, ctx->lfac);
  if (rc) return rc;
  return side_join(ctx);
}

extern "C" int dpmm_params_merge(dpmm_ctx* ctx, int64_t i, int64_t j) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  DPMM_NEED_HYPER("dpmm_params_merge");
  NEED(i >= 1 && j >= 1 && i != j && i <= ctx->Kcap_tab && j <= ctx->Kcap_tab, DPMM_EINVAL, "bad cluster pair");
  KernelTimer kt(ctx, TK_PARAMS);
  ptab_merge_kernel<<<1, 256, 0, ctx->stream>>>(ctx->ptab, ctx->stats_rec, (int)i - 1, (int)j - 1);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int dpmm_get_params_niw(dpmm_ctx* ctx, int32_t K, float* mu, double* lfac, float* logdet, float* weights,
                                   float* lr_weights) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  NEED(ctx->prior == DPMM_PRIOR_NIW, DPMM_ESTATE, "context was created with the multinomial prior");
  NEED(ctx->dev_params && ctx->params_set && K == ctx->K, DPMM_ESTATE, "no device-sampled parameters for this K");
  const int D = ctx->D;
  const size_t nrec = (size_t)3 * K;
  CK(cudaStreamSynchronize(ctx->stream));
  if (mu) CK(cudaMemcpy(mu, ctx->raw_params, nrec * D * 4, cudaMemcpyDeviceToHost));
  if (logdet) CK(cudaMemcpy(logdet, ctx->raw_params + nrec * D + nrec * D * D, nrec * 4, cudaMemcpyDeviceToHost));
  if (lfac) CK(cudaMemcpy(lfac, ctx->lfac, nrec * D * D * 8, cudaMemcpyDeviceToHost));
  if (weights) CK(cudaMemcpy(weights, ctx->w_out, (size_t)K * 4, cudaMemcpyDeviceToHost));
  if (lr_weights) CK(cudaMemcpy(lr_weights, ctx->lr_out, (size_t)2 * K * 4, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int dpmm_get_params_multinomial(dpmm_ctx* ctx, int32_t K, float* log_p, float* weights, float* lr_weights) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  NEED(ctx->prior == DPMM_PRIOR_MULTINOMIAL, DPMM_ESTATE, "context was created with the NIW prior");
  NEED(ctx->dev_params && ctx->params_set && K == ctx->K, DPMM_ESTATE, "no device-sampled parameters for this K");
  CK(cudaStreamSynchronize(ctx->stream));
  if (log_p) CK(cudaMemcpy(log_p, ctx->recs, (size_t)3 * K * ctx->D * 4, cudaMemcpyDeviceToHost));
  if (weights) CK(cudaMemcpy(weights, ctx->w_out, (size_t)K * 4, cudaMemcpyDeviceToHost));
  if (lr_weights) CK(cudaMemcpy(lr_weights, ctx->lr_out, (size_t)2 * K * 4, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int dpmm_predict_niw(dpmm_ctx* ctx, int32_t K, const float* u, const float* mu, const float* tconst,
                                const float* df, int64_t* labels, float* probs) {
  NEED(ctx && u && mu && tconst && df && labels, DPMM_EINVAL, "NULL argument");
  NEED(ctx->prior == DPMM_PRIOR_NIW, DPMM_ESTATE, "context was created with the multinomial prior");
  NEED(K >= 1 && K <= DPMM_MAX_K, DPMM_ELIMIT, "K out of range");
  CK(cudaSetDevice(ctx->device));
  const int D = ctx->D;
  const size_t nf = (size_t)K * D * D + (size_t)K * D + 2 * (size_t)K;
  float* dpar = nullptr;
  int32_t* dlab = nullptr;
  float* dprob = nullptr;
  CK(cudaMalloc((void**)&dpar, nf * 4));
  auto cleanup = [&]() {
    if (dpar) cudaFree(dpar);
    if (dlab) cudaFree(dlab);
    if (dprob) cudaFree(dprob);
  };
#define CKP(call)                                                                                        \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      cleanup();                                                                                         \
      return fail(ctx, DPMM_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                \
    }                                                                                                    \
  } while (0)
  CKP(cudaMalloc((void**)&dlab, (size_t)ctx->n * 4));
  if (probs) CKP(cudaMalloc((void**)&dprob, (size_t)ctx->n * K * 4));
  float* d_u = dpar;
  float* d_mu = d_u + (size_t)K * D * D;
  float* d_tc = d_mu + (size_t)K * D;
  float* d_df = d_tc + K;
  std::vector<float> up, mp;
  if (ctx->D_user != D) {   // padded features: unit factor rows, zero means
    const int Du = ctx->D_user;
    up.assign((size_t)K * D * D, 0.f);
    mp.assign((size_t)K * D, 0.f);
    for (int k = 0; k < K; ++k) {
      for (int i = 0; i < Du; ++i) memcpy(&up[((size_t)k * D + i) * D], u + ((size_t)k * Du + i) * Du, (size_t)Du * 4);
      for (int i = Du; i < D; ++i) up[((size_t)k * D + i) * D + i] = 1.f;
      memcpy(&mp[(size_t)k * D], mu + (size_t)k * Du, (size_t)Du * 4);
    }
    u = up.data();
    mu = mp.data();
  }
  CKP(cudaMemcpyAsync(d_u, u, (size_t)K * D * D * 4, cudaMemcpyHostToDevice, ctx->stream));
  CKP(cudaMemcpyAsync(d_mu, mu, (size_t)K * D * 4, cudaMemcpyHostToDevice, ctx->stream));
  CKP(cudaStreamSynchronize(ctx->stream));   // (the padded copies above live on this stack frame)
  CKP(cudaMemcpyAsync(d_tc, tconst, (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
  CKP(cudaMemcpyAsync(d_df, df, (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
  NiwPredictArgs pa{};
  pa.x = ctx->x; pa.n = ctx->n; pa.D = D; pa.D_true = ctx->D_user; pa.K = K; pa.u = d_u; pa.mu = d_mu; pa.tconst = d_tc; pa.df = d_df;
  pa.labels = dlab; pa.probs = dprob;
  const size_t sm = (size_t)8 * (D + K) * 4;
  if (sm > 48 * 1024) CKP(cudaFuncSetAttribute(niw_predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  {
    KernelTimer kt(ctx, TK_LABEL);
    const unsigned grid = (unsigned)std::min<int64_t>((ctx->n + 7) / 8, (int64_t)ctx->sm_count * 8);
    niw_predict_kernel<<<grid, 256, sm, ctx->stream>>>(pa);
    CKP(cudaGetLastError());
  }
  std::vector<int32_t> h((size_t)ctx->n);
  CKP(cudaMemcpyAsync(h.data(), dlab, (size_t)ctx->n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (probs) CKP(cudaMemcpyAsync(probs, dprob, (size_t)ctx->n * K * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CKP(cudaStreamSynchronize(ctx->stream));
#undef CKP
  for (int64_t i = 0; i < ctx->n; ++i) labels[i] = (int64_t)h[i] + 1;
  cleanup();
  return 0;
}

extern "C" int dpmm_predict_multinomial(dpmm_ctx* ctx, int32_t K, const double* logp, const float* logw,
                                        int64_t* labels, float* probs) {
  NEED(ctx && logp && logw && labels, DPMM_EINVAL, "NULL argument");
  NEED(ctx->prior == DPMM_PRIOR_MULTINOMIAL, DPMM_ESTATE, "context was created with the NIW prior");
  NEED(K >= 1 && K <= DPMM_MAX_K, DPMM_ELIMIT, "K out of range");
  CK(cudaSetDevice(ctx->device));
  const int D = ctx->D;
  const int64_t n = ctx->n;
  // as many clusters per tile as shared memory holds (a D = 1024 row takes 8 KB)
  const int KC = std::max(1, std::min(K, ctx->smem_optin / (D * 8)));
  const size_t sm = (size_t)KC * D * 8;
  double* dlp = nullptr;
  float* dlw = nullptr;
  float* dscore = nullptr;
  int32_t* dlab = nullptr;
  auto cleanup = [&]() {
    if (dlp) cudaFree(dlp);
    if (dlw) cudaFree(dlw);
    if (dscore) cudaFree(dscore);
    if (dlab) cudaFree(dlab);
  };
#define CKP(call)                                                                                        \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      cleanup();                                                                                         \
      return fail(ctx, DPMM_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                \
    }                                                                                                    \
  } while (0)
  CKP(cudaMalloc((void**)&dlp, (size_t)K * D * 8));
  CKP(cudaMalloc((void**)&dlw, (size_t)K * 4));
  CKP(cudaMalloc((void**)&dscore, (size_t)n * K * 4));
  CKP(cudaMalloc((void**)&dlab, (size_t)n * 4));
  CKP(cudaMemcpyAsync(dlp, logp, (size_t)K * D * 8, cudaMemcpyHostToDevice, ctx->stream));
  CKP(cudaMemcpyAsync(dlw, logw, (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
  MnmScoreArgs sa{};
  sa.x = ctx->x; sa.n = n; sa.D = D; sa.K = K; sa.KC = KC; sa.logp = dlp; sa.logw = dlw; sa.score = dscore;
  if (sm > 48 * 1024) CKP(cudaFuncSetAttribute(mnm_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  {
    KernelTimer kt(ctx, TK_LABEL, 2);
    const unsigned gx = (unsigned)std::min<int64_t>((n + 7) / 8, (int64_t)ctx->sm_count * 8);
    mnm_score_kernel<<<dim3(gx, (unsigned)((K + KC - 1) / KC)), 256, sm, ctx->stream>>>(sa);
    CKP(cudaGetLastError());
    mnm_predict_finish_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0,
                                ctx->stream>>>(dscore, n, K, dlab, probs != nullptr);
    CKP(cudaGetLastError());
  }
  std::vector<int32_t> h((size_t)n);
  CKP(cudaMemcpyAsync(h.data(), dlab, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (probs) CKP(cudaMemcpyAsync(probs, dscore, (size_t)n * K * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CKP(cudaStreamSynchronize(ctx->stream));
#undef CKP
  for (int64_t i = 0; i < n; ++i) labels[i] = (int64_t)h[i] + 1;
  cleanup();
  return 0;
}

extern "C" int dpmm_debug_loglik(dpmm_ctx* ctx, int32_t which, float* out) {
  NEED(ctx && out, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  NEED(ctx->params_set, DPMM_ESTATE, "set_params must precede debug_loglik");
  NEED(which == 0 || which == 1, DPMM_EINVAL, "which must be 0 or 1");
  const size_t cols = which == 0 ? (size_t)ctx->K : 2;
  float* dump = nullptr;
  CK(cudaMalloc((void**)&dump, cols * ctx->n * 4));
  int rc = 0;
  if (which == 0) {
    // a dry run of the label kernel on a scratch label array: state (labels, RNG counter) untouched
    int32_t* keep = ctx->labels;
    int32_t* scratch = nullptr;
    const uint32_t call0 = ctx->call;
    const int lb0 = ctx->label_bound;
    if (cudaMalloc((void**)&scratch, (size_t)ctx->n * 4) != cudaSuccess) {
      cudaFree(dump);
      return fail(ctx, DPMM_ECUDA, "cudaMalloc(scratch labels) failed");
    }
    ctx->labels = scratch;
    rc = run_sample_labels(ctx, 1, dump);
    cudaStreamSynchronize(ctx->stream);
    ctx->labels = keep;
    ctx->call = call0;
    ctx->label_bound = lb0;
    ctx->hist_valid = ctx->scan_valid = ctx->sorted = ctx->partitioned = ctx->stats_cached = false;  // the histogram describes the scratch labels
    cudaFree(scratch);
  } else {
    // sub-label matrix under the CURRENT labels; sub-labels are restored afterwards
    uint8_t* keep = nullptr;
    const uint32_t call0 = ctx->call;
    if (ctx->label_bound > ctx->K) {
      cudaFree(dump);
      return fail(ctx, DPMM_ESTATE, "labels refer to clusters beyond the K of set_params");
    }
    if (cudaMalloc((void**)&keep, (size_t)ctx->n) != cudaSuccess) {
      cudaFree(dump);
      return fail(ctx, DPMM_ECUDA, "cudaMalloc(scratch sub-labels) failed");
    }
    cudaMemcpyAsync(keep, ctx->sub, (size_t)ctx->n, cudaMemcpyDeviceToDevice, ctx->stream);
    rc = run_sublabels(ctx, true, dump);
    cudaMemcpyAsync(ctx->sub, keep, (size_t)ctx->n, cudaMemcpyDeviceToDevice, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    ctx->call = call0;
    ctx->partitioned = ctx->stats_cached = false;
    cudaFree(keep);
  }
  if (rc == 0) {
    cudaError_t e = cudaMemcpy(out, dump, cols * ctx->n * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(ctx, DPMM_ECUDA, std::string("cudaMemcpy(dump): ") + cudaGetErrorString(e));
  }
  cudaFree(dump);
  return rc;
}

extern "C" int dpmm_debug_tc_stats(dpmm_ctx* ctx, int64_t* out3) {
  NEED(ctx && out3, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  out3[0] = out3[1] = out3[2] = 0;
  if (ctx->tc_stats == nullptr) return 0;
  int32_t h[2] = {0, 0};
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(h, ctx->tc_stats, 8, cudaMemcpyDeviceToHost));
  out3[0] = h[0];
  out3[1] = h[1];
  if (ctx->t2_ctr != nullptr) {
    CK(cudaMemcpy(h, ctx->t2_ctr, 4, cudaMemcpyDeviceToHost));
    out3[2] = h[0];
  }
  return 0;
}

extern "C" int dpmm_debug_sort(dpmm_ctx* ctx, int32_t* perm, int64_t* moved) {
  NEED(ctx && moved, DPMM_EINVAL, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  moved[0] = 0;
  if (perm != nullptr) {
    int rc = ensure_sorted(ctx);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  if (perm != nullptr) CK(cudaMemcpy(perm, ctx->perm, (size_t)ctx->n * 4, cudaMemcpyDeviceToHost));
  if (ctx->ctr_sets != nullptr) {
    int32_t h = 0;
    CK(cudaMemcpy(&h, ctx->tc_stats + 4, 4, cudaMemcpyDeviceToHost));
    moved[0] = h;
  }
  return 0;
}

extern "C" int dpmm_debug_fused_stats(dpmm_ctx* ctx, int64_t* out3) {
  NEED(ctx && out3, DPMM_EINVAL, "NULL argument");
  out3[0] = ctx->n_fused;
  out3[1] = ctx->n_cached;
  out3[2] = ctx->n_recompute;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// timing hooks
// ------------------------------------------------------------------------------------------------
extern "C" int dpmm_timing_kinds(void) { return TK_COUNT; }
extern "C" const char* dpmm_timing_name(int32_t kind) { return (kind >= 0 && kind < TK_COUNT) ? kTimingNames[kind] : ""; }
extern "C" int64_t dpmm_launch_count(const dpmm_ctx* ctx) { return ctx ? ctx->launches : 0; }

static void drain_timers(dpmm_ctx* ctx) {
  for (auto& t : ctx->tev) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) ctx->t_ms[t.kind] += ms;
    ctx->ev_pool.push_back(t.a);
    ctx->ev_pool.push_back(t.b);
  }
  ctx->tev.clear();
}

extern "C" int dpmm_timing_enable(dpmm_ctx* ctx, int32_t on) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  drain_timers(ctx);
  ctx->timing = on != 0;
  return 0;
}

extern "C" int dpmm_timing_read(dpmm_ctx* ctx, double* ms, int64_t* launches, int32_t reset) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  drain_timers(ctx);
  for (int k = 0; k < TK_COUNT; ++k) {
    if (ms) ms[k] = ctx->t_ms[k];
    if (launches) launches[k] = ctx->t_n[k];
    if (reset) {
      ctx->t_ms[k] = 0;
      ctx->t_n[k] = 0;
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// NCCL (resolved at run time so that single-GPU users need no NCCL at all)
// ------------------------------------------------------------------------------------------------
static int load_nccl(dpmm_ctx* ctx, NcclApi& api) {
  if (api.handle) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (api.handle) break;
  }
  if (!api.handle) return fail(ctx, DPMM_ENCCL, std::string("dlopen(libnccl.so.2) failed: ") + dlerror());
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
  api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
  api.AllGather = (decltype(api.AllGather))dlsym(api.handle, "ncclAllGather");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy || !api.GetErrorString)
    return fail(ctx, DPMM_ENCCL, "libnccl is missing a required symbol");
  return 0;
}

extern "C" int dpmm_nccl_unique_id(void* out128) {
  dpmm_ctx* ctx = nullptr;
  NEED(out128, DPMM_EINVAL, "out128 is NULL");
  static NcclApi api;
  int rc = load_nccl(nullptr, api);
  if (rc) return rc;
  const int r = api.GetUniqueId(out128);
  if (r != 0) return fail(nullptr, DPMM_ENCCL, std::string("ncclGetUniqueId: ") + api.GetErrorString(r));
  return 0;
}

extern "C" int dpmm_comm_init(dpmm_ctx* ctx, const void* unique_id128, int32_t rank, int32_t world_size) {
  NEED(ctx && unique_id128, DPMM_EINVAL, "NULL argument");
  NEED(world_size >= 1 && rank >= 0 && rank < world_size, DPMM_EINVAL, "bad rank / world size");
  CK(cudaSetDevice(ctx->device));
  int rc = load_nccl(ctx, ctx->nccl);
  if (rc) return rc;
  UidBlob id;
  memcpy(id.b, unique_id128, 128);
  const int r = ctx->nccl.CommInitRank(&ctx->comm, world_size, id, rank);
  if (r != 0) return fail(ctx, DPMM_ENCCL, std::string("ncclCommInitRank: ") + ctx->nccl.GetErrorString(r));
  ctx->world = world_size;
  ctx->rank = rank;
  // ---- peer-memory exchange regions (optional: any failure leaves the NCCL all-reduce in charge) ----
  if (world_size > 1 && world_size <= IPC_MAX_WORLD && ctx->nccl.AllGather && env_int("DPMM_ALLREDUCE_IPC", 1) != 0) {
    const size_t cap = ((size_t)32 << 20) / 8;   // 32 MB per buffer
    const size_t bytes = IPC_FLAG_BYTES + 2 * cap * 8;
    cudaIpcMemHandle_t mine;
    char* hbuf = nullptr;
    bool ok = cudaMalloc((void**)&ctx->ipc_local, bytes) == cudaSuccess && cudaMemset(ctx->ipc_local, 0, bytes) == cudaSuccess &&
              cudaIpcGetMemHandle(&mine, ctx->ipc_local) == cudaSuccess &&
              cudaMalloc((void**)&hbuf, (size_t)(world_size + 1) * sizeof(mine)) == cudaSuccess;
    std::vector<cudaIpcMemHandle_t> all(world_size);
    if (ok) {
      ok = cudaMemcpy(hbuf + (size_t)world_size * sizeof(mine), &mine, sizeof(mine), cudaMemcpyHostToDevice) == cudaSuccess &&
           ctx->nccl.AllGather(hbuf + (size_t)world_size * sizeof(mine), hbuf, sizeof(mine), /*ncclChar*/ 0, ctx->comm, ctx->stream) == 0 &&
           cudaStreamSynchronize(ctx->stream) == cudaSuccess &&
           cudaMemcpy(all.data(), hbuf, (size_t)world_size * sizeof(mine), cudaMemcpyDeviceToHost) == cudaSuccess;
    }
    int nopen = 0;
    for (int p = 0; ok && p < world_size; ++p) {
      if (p == rank) continue;
      ok = cudaIpcOpenMemHandle((void**)&ctx->ipc_peer[p], all[p], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      if (ok) ++nopen;
    }
    if (hbuf) cudaFree(hbuf);
    // every rank must take the same path: agree through one more collective (sum of the ok flags)
    double* agree = nullptr;
    int all_ok = 0;
    if (cudaMalloc((void**)&agree, 8) == cudaSuccess) {
      const double v = ok ? 1.0 : 0.0;
      double got = 0.0;
      if (cudaMemcpy(agree, &v, 8, cudaMemcpyHostToDevice) == cudaSuccess &&
          ctx->nccl.AllReduce(agree, agree, 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0, ctx->comm, ctx->stream) == 0 &&
          cudaStreamSynchronize(ctx->stream) == cudaSuccess && cudaMemcpy(&got, agree, 8, cudaMemcpyDeviceToHost) == cudaSuccess)
        all_ok = (int)llround(got) == world_size;
      cudaFree(agree);
    }
    cudaGetLastError();   // a failed optional step must not poison later calls
    ctx->ipc_ok = all_ok != 0;
    ctx->ipc_cap = cap;
    if (env_int("DPMM_VERBOSE", 0))
      fprintf(stderr, "[dpmm] rank %d: peer-memory all-reduce %s (%d peers mapped)\n", rank, ctx->ipc_ok ? "enabled" : "unavailable, using NCCL", nopen);
  }
  return 0;
}
