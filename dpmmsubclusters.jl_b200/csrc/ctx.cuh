// Context, error plumbing and per-launch timing shared by the translation units of libdpmm_b200.so.
#pragma once
#include "../../include/dpmm_b200.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

struct StatsItem;
struct SmartState;   // smart.cu

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
enum TimingKind {
  TK_LABEL = 0,     // fused log-likelihood + label draw
  TK_SORT,          // histogram / scan / scatter
  TK_SUBLABEL,      // sub-label draw + left/right partition
  TK_STATS,         // segmented sufficient statistics
  TK_STATS_AUX,     // work list + finalise/pack
  TK_RELABEL,       // LUT relabel / init
  TK_ALLREDUCE,     // NCCL all-reduce of the packed statistics
  TK_LABEL_OVF,     // full-K overflow kernel of the D = 32 / 64 tensor-core label path
  TK_PARAMS,        // parameter packing / device-side parameter step
  TK_COUNT
};
static const char* const kTimingNames[TK_COUNT] = {"label", "sort", "sublabel", "stats", "stats_aux", "relabel", "allreduce", "label_ovf", "params"};

struct TimedEvent {
  cudaEvent_t a, b;
  int kind;
};

struct UidBlob {  // layout of ncclUniqueId (128 opaque bytes, passed by value)
  char b[128];
};
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, UidBlob, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
struct dpmm_ctx {
  int device = 0;
  int sm_count = 148;
  int smem_optin = 0;
  int smem_per_sm = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  // side stream of the device parameter step: kernels that do not depend on each other (mixture weights next to the
  // Bartlett draws, the K x K merge table next to the posteriors) run on it between a fork and a join event
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int64_t n = 0;
  int D = 0;        // feature dimension the kernels run at (D_user zero-padded to an instantiated width)
  int D_user = 0;   // feature dimension at the boundary
  int prior = 0;
  uint64_t seed = 0;
  int64_t goff = 0;
  uint32_t call = 0;
  int sampler = 0;
  std::string err;

  float* x = nullptr;              // dense points [n][D]; NULL for a sparse context
  // sparse context (dpmm_create_sparse, multinomial): the points as compressed rows, see kernels_mnm_sparse.cuh
  bool sparse = false;
  int64_t nnz = 0;
  int64_t* sp_ptr = nullptr;       // [n + 1]
  int32_t* sp_idx = nullptr;       // [nnz]
  float* sp_val = nullptr;         // [nnz]
  int32_t* labels = nullptr;
  uint8_t* sub = nullptr;
  int32_t* perm = nullptr;
  int32_t* perm2 = nullptr;
  int64_t* wide = nullptr;         // [n] scratch of the boundary conversions (1-based Int64 <-> device types)
  int32_t* wide_status = nullptr;
  double* u_label = nullptr;
  double* u_sub = nullptr;
  uint8_t* r_bits = nullptr;

  // K-sized state
  int K = 0, Kcap = 0;    // K = number of clusters of the last set_params
  int label_bound = 1;    // every label value is < label_bound (0-based)
  bool params_set = false;
  int rec_f = 0;          // floats per distribution record (NIW) / D (multinomial)
  float* raw_params = nullptr;  // NIW: [3K](mu[D] | invSigma[D][D] | logdet) as uploaded, input of niw_pack_kernel
  float* recs = nullptr;  // [3K][rec_f]
  float* cst = nullptr;   // [3K]
  float* logw = nullptr;  // [K]
  float* loglr = nullptr; // [2K]
  // tensor-core label path (NIW, D == 32): stacked K-major factors, U mu, mu, |U|_F, TMA descriptor of X
  float* tc_w = nullptr;
  float* tc_b = nullptr;
  float* tc_mu = nullptr;
  float* tc_fro = nullptr;
  int32_t* tc_stats = nullptr;
  // second-generation tensor-core label path (NIW, D == 32 or 64): operand images, rows of U, overflow counter
  float* t2_piv = nullptr;
  float* t2_scr = nullptr;
  float* t2_u = nullptr;
  float* t2_bias = nullptr;
  float* t2_fro8 = nullptr;
  int32_t* t2_ctr = nullptr;
  int32_t* ctr_sets = nullptr;   // [2][T2_CTR_SET]: tc_stats / t2_ctr point into the set of the current label call
  int ctr_cur = 0;
  bool ctr_clean = false;        // the set the next tensor-core label call takes is known to be zero
  bool t2_ok = false;       // shape supported
  bool t2_params = false;   // t2_* describe the current parameters
  int t2_KS = 0, t2_nch = 0;
  // adaptive path choice: counters of the last tensor-core label call (points, exact evaluations, overflow points)
  // land in pinned memory behind an event; a call that finds more exact work than the FMA kernel would do for all K
  // clusters sends the next calls to the FMA kernel for a while (early iterations, heavily overlapping clusters)
  int32_t* t2_hstat = nullptr;       // mapped pinned [4], written by the overflow kernel's last block
  int32_t* t2_hstat_dev = nullptr;   // its device address
  cudaEvent_t t2_hstat_ev = nullptr;
  bool t2_hstat_pending = false;
  int t2_cooldown = 0;
  // fused sub-label + statistics tensor-core path (NIW, D == 32): U rows / bias / centre per cluster, left counts
  float* ss_w = nullptr;
  float* ss_b = nullptr;
  float* ss_c = nullptr;
  int32_t* lcount = nullptr;
  CUtensorMap tmap_x;
  float* mtc_w = nullptr;   // multinomial tensor-core path: TF32-exact 3-way split of the log-probabilities
  bool mtc_ok = false;      // multinomial: tensor map built and the counts are TF32-exact
  bool mtc_params = false;
  bool tc_ok = false;       // tensor map built
  bool tc_params = false;   // tc_* describe the current parameters
  float* logp_t = nullptr;  // multinomial [D][KP]
  int KP = 0;
  // label histograms: two buffers of Kcap entries.  A tensor-core label call fills one (ctx->hist from then on) while
  // its overflow kernel clears the other for the next call, so no memset sits between the sweeps
  int32_t* hist_mem = nullptr;
  int32_t* hist = nullptr;        // the buffer of the current labels
  int hist_cur = 0;
  int hist_spare_clean = 0;       // entries of the other buffer known to be zero
  // moved-point counter of the last tensor-core label call, while perm still sorts the labels that call started from
  // and nothing else changed them: the sort after it then skips the scatter when the counter is 0
  const int32_t* t2_moved = nullptr;
  int risk_zeroed_k = 0;          // K > 0: the label scatter cleared the risk slot outbuf[3 K rec] (no memset before the finalise)
  int pdl_tmem = -1;              // tensor memory may be allocated before the grid dependency (sweep_pdl_ok); -1: not checked yet
  int32_t* seg_off = nullptr;
  int32_t* scat_cursor = nullptr;
  int32_t* lr_cursor = nullptr;
  int32_t* lut_l = nullptr;
  int32_t* lut_r = nullptr;
  uint8_t* rule = nullptr;
  uint8_t* wanted = nullptr;
  int32_t* idx_list = nullptr;
  int stats_rec = 0;
  double* acc = nullptr;
  float* centers = nullptr;   // [2K][D] per-run shift of the tensor-core statistics
  double* outbuf = nullptr;
  StatsItem* items = nullptr;
  int64_t items_cap = 0;
  int32_t* item_ctr = nullptr;  // [0]=n_items [1]=next_item
  int chunk = 1024;

  // pinned staging: hstage for results coming back (the call synchronises anyway); two alternating upload
  // buffers, each guarded by an event recorded after its last copy, so that an upload never waits for the stream
  void* hstage = nullptr;
  size_t hstage_bytes = 0;
  void* hup[2] = {nullptr, nullptr};
  size_t hup_bytes[2] = {0, 0};
  cudaEvent_t hup_ev[2] = {nullptr, nullptr};
  int hup_i = 0;

  bool hist_valid = false, sorted = false, partitioned = false;
  bool scan_valid = false;     // seg_off / scatter cursors / left-right cursors already hold the scan of `hist`
  int64_t n_fused = 0, n_cached = 0, n_recompute = 0;   // DPMM_VERBOSE counters
  bool acc_cleared = false;    // acc / lcount were zeroed by the last label scatter and not touched since
  bool stats_cached = false;   // acc / lcount / centers hold the l/r statistics of every cluster for the current labels
  bool cursors_fresh = false;  // lr_cursor still holds the segment bounds (not yet consumed by a partition)
  int64_t launches = 0;
  bool timing = false;
  std::vector<TimedEvent> tev;
  std::vector<cudaEvent_t> ev_pool;
  double t_ms[TK_COUNT] = {0};
  int64_t t_n[TK_COUNT] = {0};

  // device-side parameter step (NIW): hyper-parameters, persistent statistics / posterior tables, factors
  bool dev_params = false;
  double alpha = 0.0;
  double* hyper_d = nullptr;     // [NIW_HYPER_DOUBLES(D_user)]
  double* ptab = nullptr;        // [Kcap][3][stats_rec]   (records at D)
  double* ptab_alt = nullptr;
  double* post = nullptr;        // [Kcap][3][NIW_POST_DOUBLES(D_user)]
  double* post_alt = nullptr;
  double* lfac = nullptr;        // [3 Kcap][D][D]   (padded features: identity rows / columns)
  double* pm_out = nullptr;      // [Kcap*3*2 + Kcap*Kcap + 2] results of the posterior step for the host
  uint8_t* splittable_d = nullptr;
  int32_t* newof_d = nullptr;
  float* w_out = nullptr;        // [Kcap] Float32 mixture weights of the last dpmm_sample_params
  float* lr_out = nullptr;       // [2 Kcap]
  uint32_t pcall = 0;
  int Kcap_tab = 0;

  SmartState* smart = nullptr;   // buffers of the smart-split worker functions (smart.cu)

  NcclApi nccl;
  void* comm = nullptr;
  int world = 1, rank = 0;
  // one-shot all-reduce of the packed statistics over peer memory (NVLink): every rank maps every peer's
  // exchange region [flags | buffer 0 | buffer 1] through CUDA IPC; see kernels_ipc.cuh
  bool ipc_ok = false;
  uint8_t* ipc_local = nullptr;
  uint8_t* ipc_peer[16] = {nullptr};
  size_t ipc_cap = 0;        // doubles per buffer
  uint32_t ipc_epoch = 0;
};

void dpmm_internal_smart_free(dpmm_ctx* ctx);      // smart.cu
int dpmm_internal_ensure_sorted(dpmm_ctx* ctx);    // dpmm_b200.cu

inline thread_local std::string g_err;

inline int fail(dpmm_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  g_err = msg;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(ctx, DPMM_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));          \
  } while (0)
#define NEED(cond, code, msg) \
  do {                        \
    if (!(cond)) return fail(ctx, code, msg); \
  } while (0)

struct KernelTimer {
  dpmm_ctx* c;
  cudaEvent_t a = nullptr, b = nullptr;
  int kind;
  KernelTimer(dpmm_ctx* c_, int kind_, int nlaunch = 1) : c(c_), kind(kind_) {
    c->launches += nlaunch;
    if (c->timing) {
      auto get = [&]() {
        cudaEvent_t e;
        if (!c->ev_pool.empty()) {
          e = c->ev_pool.back();
          c->ev_pool.pop_back();
        } else {
          cudaEventCreate(&e);
        }
        return e;
      };
      a = get();
      b = get();
      cudaEventRecord(a, c->stream);
    }
  }
  ~KernelTimer() {
    if (a) {
      cudaEventRecord(b, c->stream);
      c->tev.push_back(TimedEvent{a, b, kind});
      c->t_n[kind] += 1;
    }
  }
};

// fork: `side` waits for everything enqueued on the main stream so far; join: the main stream waits for `side`
inline int side_fork(dpmm_ctx* ctx) {
  if (ctx->side == nullptr) {
    CK(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  }
  CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  CK(cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0));
  return 0;
}
inline int side_join(dpmm_ctx* ctx) {
  CK(cudaEventRecord(ctx->ev_join, ctx->side));
  CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  return 0;
}

inline int ensure_stage(dpmm_ctx* ctx, size_t bytes) {
  if (ctx->hstage_bytes >= bytes) return 0;
  if (ctx->hstage) cudaFreeHost(ctx->hstage);
  ctx->hstage = nullptr;
  ctx->hstage_bytes = 0;
  size_t want = std::max(bytes, (size_t)1 << 20);
  CK(cudaMallocHost(&ctx->hstage, want));
  ctx->hstage_bytes = want;
  return 0;
}

// Next upload staging buffer (>= bytes): waits only for the copies issued from THIS buffer two uploads ago.
inline int upload_acquire(dpmm_ctx* ctx, size_t bytes, void** out) {
  const int i = ctx->hup_i;
  ctx->hup_i ^= 1;
  if (ctx->hup_ev[i] == nullptr) CK(cudaEventCreateWithFlags(&ctx->hup_ev[i], cudaEventDisableTiming));
  CK(cudaEventSynchronize(ctx->hup_ev[i]));
  if (ctx->hup_bytes[i] < bytes) {
    if (ctx->hup[i]) cudaFreeHost(ctx->hup[i]);
    ctx->hup[i] = nullptr;
    ctx->hup_bytes[i] = 0;
    const size_t want = std::max(bytes, (size_t)1 << 20);
    CK(cudaMallocHost(&ctx->hup[i], want));
    ctx->hup_bytes[i] = want;
  }
  *out = ctx->hup[i];
  return i;
}
inline int upload_release(dpmm_ctx* ctx, int i) {
  CK(cudaEventRecord(ctx->hup_ev[i], ctx->stream));
  return 0;
}

template <typename T>
inline cudaError_t dev_realloc(T** p, size_t count) {
  if (*p) cudaFree(*p);
  *p = nullptr;
  return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
}

// number of label values any K-sized table must cover
inline int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

// NIW feature dimensions with instantiated kernels, grouped into the translation units
// launch_niw.cu is compiled into (DPMM_DIMSET = 0..5)
#define DPMM_NIW_NSETS 6
int niw_launch_label(dpmm_ctx* ctx, const struct GaussLabelArgs& a);
int niw_launch_sublabel(dpmm_ctx* ctx, const struct SubLabelArgs& a, bool sample);
int niw_launch_stats(dpmm_ctx* ctx, const struct StatsArgs& a);
