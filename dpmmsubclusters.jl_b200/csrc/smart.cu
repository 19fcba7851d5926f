// Smart splits, worker side (SURVEY.md 8f-3): the three worker functions smart_cluster_init! drives
//   tranform_points_worker!       src/local_clusters_actions.jl:641-652   t = v'(x - mu) of one cluster + two percentiles
//   kmeans_iter_worker!           :633-639                                1-D 2-means assignment + per-side (sum, count)
//   set_smart_labels_in_worker!   :627-631                                sub-labels of the cluster <- the assignment
// and the master's reductions over the workers (:578-613: minimum / maximum of the percentiles, sums of the
// per-side sums and counts), which run here as small NCCL all-reduces when a communicator is attached.
//
// Arithmetic follows the reference: `pts[:, mask] .- mu` promotes the Float32 points to Float64 (mu = points_sum / N
// is Float64), so the projection, the percentiles and the sums are Float64.  percentile(t, p) is StatsBase's
// quantile(t, p / 100) -- the reference passes 0.10 and 0.90, i.e. the 0.1 % and 0.9 % quantiles -- with Julia's
// default definition (type 7): h = (n - 1) q + 1, t_(floor h) + (h - floor h)(t_(floor h + 1) - t_(floor h)).
// The order statistics come from a device radix sort (CUB) of the projected values.  The per-side sums are
// reduced in a fixed order (per-block partials summed on the host), so a call is reproducible.
#include "ctx.cuh"
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <limits>

struct SmartState {
  int cluster = -1;        // 0-based cluster the buffers describe
  int beg = 0, cnt = 0;    // its segment of ctx->perm
  double* t = nullptr;     // [cap] projected values, segment order
  double* ts = nullptr;    // [cap] sorted
  uint8_t* lab = nullptr;  // [cap] 0 = nearer to min_mean, 1 = nearer to max_mean
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
  int cap = 0;
  double* vmu = nullptr;   // [2 D] device
  double* part = nullptr;  // [SMART_BLOCKS][4] per-block partials
  double* red = nullptr;   // [8] all-reduce scratch
  bool assigned = false;
};
#define SMART_BLOCKS 592
#define SMART_THREADS 256

__global__ void __launch_bounds__(SMART_THREADS) smart_project_kernel(const float* __restrict__ x, int D, int Du,
                                                                      const int32_t* __restrict__ perm, int beg, int cnt,
                                                                      const double* __restrict__ vmu, double* __restrict__ t) {
  extern __shared__ double sm_v[];   // v | mu
  for (int e = threadIdx.x; e < 2 * Du; e += blockDim.x) sm_v[e] = vmu[e];
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) {
    const float* row = x + (size_t)perm[beg + i] * D;
    double acc = 0.0;
    for (int d = 0; d < Du; ++d) acc += sm_v[d] * ((double)__ldg(row + d) - sm_v[Du + d]);
    t[i] = acc;
  }
}

__global__ void __launch_bounds__(SMART_THREADS) smart_kmeans_kernel(const double* __restrict__ t, int cnt, double mn, double mx,
                                                                     uint8_t* __restrict__ lab, double* __restrict__ part) {
  double s0 = 0.0, s1 = 0.0, c0 = 0.0, c1 = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) {
    const double v = t[i];
    const bool lo = fabs(v - mn) < fabs(v - mx);   // kmeans_iter_worker!: abs(x - min_mean) < abs(x - max_mean) ? 1 : 2
    lab[i] = lo ? 0 : 1;
    if (lo) { s0 += v; c0 += 1.0; } else { s1 += v; c1 += 1.0; }
  }
  __shared__ double red[4][SMART_THREADS / 32];
  double vals[4] = {s0, c0, s1, c1};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    double v = vals[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double v = 0.0;
    for (int w = 0; w < SMART_THREADS / 32; ++w) v += red[threadIdx.x][w];
    part[blockIdx.x * 4 + threadIdx.x] = v;
  }
}

__global__ void __launch_bounds__(SMART_THREADS) smart_set_kernel(const int32_t* __restrict__ perm, int beg, int cnt,
                                                                  const uint8_t* __restrict__ lab, uint8_t* __restrict__ sub) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) sub[perm[beg + i]] = lab[i];
}

void dpmm_internal_smart_free(dpmm_ctx* ctx) {
  SmartState* s = ctx->smart;
  if (!s) return;
  cudaFree(s->t); cudaFree(s->ts); cudaFree(s->lab); cudaFree(s->tmp); cudaFree(s->vmu); cudaFree(s->part); cudaFree(s->red);
  delete s;
  ctx->smart = nullptr;
}

static unsigned smart_grid(int cnt) { return (unsigned)std::max(1, std::min((cnt + SMART_THREADS - 1) / SMART_THREADS, SMART_BLOCKS)); }

// all-reduce of n <= 8 doubles held on the host; op: 0 = sum, 2 = max (ncclRedOp_t)
static int smart_allreduce(dpmm_ctx* ctx, SmartState* s, double* h, int n, int op) {
  if (ctx->comm == nullptr || ctx->world <= 1) return 0;
  CK(cudaMemcpyAsync(s->red, h, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  const int r = ctx->nccl.AllReduce(s->red, s->red, (size_t)n, /*ncclFloat64*/ 8, op, ctx->comm, ctx->stream);
  if (r != 0) return fail(ctx, DPMM_ENCCL, std::string("ncclAllReduce: ") + ctx->nccl.GetErrorString(r));
  CK(cudaMemcpyAsync(h, s->red, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dpmm_smart_project(dpmm_ctx* ctx, int64_t cluster, const double* v, const double* mu, double* lo_hi,
                                  int64_t* count) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(v && mu && lo_hi && count, DPMM_EINVAL, "NULL argument");
  NEED(cluster >= 1 && cluster <= DPMM_MAX_K, DPMM_EINVAL, "cluster index out of range");
  NEED(ctx->x != nullptr, DPMM_ESTATE, "smart splits project the dense points: a sparse context has none");
  NEED(ctx->prior != DPMM_PRIOR_DIAG_GAUSSIAN, DPMM_ESTATE, "smart splits need the full scatter matrix: not on a diagonal context");
  CK(cudaSetDevice(ctx->device));
  if (!ctx->smart) ctx->smart = new SmartState();
  SmartState* s = ctx->smart;
  s->cluster = -1;
  s->assigned = false;
  int rc = dpmm_internal_ensure_sorted(ctx);
  if (rc) return rc;
  const int Du = ctx->D_user, D = ctx->D;
  const int c = (int)cluster - 1;
  int32_t seg[2] = {0, 0};
  if (c < std::max(std::max(ctx->K, ctx->label_bound), 1)) {
    CK(cudaMemcpyAsync(seg, ctx->seg_off + c, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  const int cnt = seg[1] - seg[0];
  if (!s->vmu) {
    CK(cudaMalloc((void**)&s->vmu, (size_t)2 * Du * 8));
    CK(cudaMalloc((void**)&s->part, (size_t)SMART_BLOCKS * 4 * 8));
    CK(cudaMalloc((void**)&s->red, 8 * 8));
  }
  if (cnt > s->cap) {
    cudaFree(s->t); cudaFree(s->ts); cudaFree(s->lab); cudaFree(s->tmp);
    s->t = s->ts = nullptr; s->lab = nullptr; s->tmp = nullptr; s->cap = 0;
    const int cap = std::max(cnt, 1024);
    CK(cudaMalloc((void**)&s->t, (size_t)cap * 8));
    CK(cudaMalloc((void**)&s->ts, (size_t)cap * 8));
    CK(cudaMalloc((void**)&s->lab, (size_t)cap));
    size_t tb = 0;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, s->t, s->ts, cap, 0, 64, ctx->stream));
    CK(cudaMalloc(&s->tmp, std::max<size_t>(tb, 16)));
    s->tmp_bytes = tb;
    s->cap = cap;
  }
  double local[2] = {-std::numeric_limits<double>::infinity(), -std::numeric_limits<double>::infinity()};   // {-lo, hi}
  if (cnt > 0) {
    std::vector<double> h(2 * Du);
    for (int d = 0; d < Du; ++d) { h[d] = v[d]; h[Du + d] = mu[d]; }
    CK(cudaMemcpyAsync(s->vmu, h.data(), (size_t)2 * Du * 8, cudaMemcpyHostToDevice, ctx->stream));
    {
      KernelTimer kt(ctx, TK_RELABEL);
      smart_project_kernel<<<smart_grid(cnt), SMART_THREADS, (size_t)2 * Du * 8, ctx->stream>>>(ctx->x, D, Du, ctx->perm, seg[0], cnt,
                                                                                               s->vmu, s->t);
      CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(ctx->stream));   // h is read by the copy above
    if (cnt > 1) {   // tranform_points_worker!: `if length(transformed_pts) > 1`
      size_t tb = s->tmp_bytes;
      {
        KernelTimer kt(ctx, TK_RELABEL, 3);
        CK(cub::DeviceRadixSort::SortKeys(s->tmp, tb, s->t, s->ts, cnt, 0, 64, ctx->stream));
      }
      const double qs[2] = {0.10 / 100.0, 0.90 / 100.0};
      double q[2];
      for (int a = 0; a < 2; ++a) {
        const double aleph = (double)cnt * qs[a] + (1.0 - qs[a]);
        const int j = std::min(std::max((int)aleph, 1), cnt - 1);
        const double g = std::min(std::max(aleph - (double)j, 0.0), 1.0);
        double ab[2];
        CK(cudaMemcpyAsync(ab, s->ts + (j - 1), 16, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        q[a] = ab[0] + g * (ab[1] - ab[0]);
      }
      local[0] = -q[0];
      local[1] = q[1];
    }
  }
  double cg = (double)cnt;
  rc = smart_allreduce(ctx, s, local, 2, /*ncclMax*/ 2);
  if (rc) return rc;
  rc = smart_allreduce(ctx, s, &cg, 1, /*ncclSum*/ 0);
  if (rc) return rc;
  const bool any = local[1] != -std::numeric_limits<double>::infinity();
  lo_hi[0] = any ? -local[0] : std::numeric_limits<double>::quiet_NaN();
  lo_hi[1] = any ? local[1] : std::numeric_limits<double>::quiet_NaN();
  *count = (int64_t)cg;
  s->cluster = c;
  s->beg = seg[0];
  s->cnt = cnt;
  return 0;
}

extern "C" int dpmm_smart_kmeans_iter(dpmm_ctx* ctx, double min_mean, double max_mean, double* out4) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  NEED(out4, DPMM_EINVAL, "NULL argument");
  SmartState* s = ctx->smart;
  NEED(s && s->cluster >= 0, DPMM_ESTATE, "dpmm_smart_kmeans_iter needs a preceding dpmm_smart_project");
  NEED(ctx->sorted, DPMM_ESTATE, "labels changed since dpmm_smart_project");
  CK(cudaSetDevice(ctx->device));
  double tot[4] = {0.0, 0.0, 0.0, 0.0};   // sum_1, count_1, sum_2, count_2
  if (s->cnt > 0) {
    const unsigned grid = smart_grid(s->cnt);
    {
      KernelTimer kt(ctx, TK_RELABEL);
      smart_kmeans_kernel<<<grid, SMART_THREADS, 0, ctx->stream>>>(s->t, s->cnt, min_mean, max_mean, s->lab, s->part);
      CK(cudaGetLastError());
    }
    int rc = ensure_stage(ctx, (size_t)SMART_BLOCKS * 4 * 8);
    if (rc) return rc;
    double* hp = static_cast<double*>(ctx->hstage);
    CK(cudaMemcpyAsync(hp, s->part, (size_t)grid * 4 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (unsigned b = 0; b < grid; ++b)
      for (int q = 0; q < 4; ++q) tot[q] += hp[b * 4 + q];
  }
  int rc = smart_allreduce(ctx, s, tot, 4, /*ncclSum*/ 0);
  if (rc) return rc;
  for (int q = 0; q < 4; ++q) out4[q] = tot[q];
  s->assigned = true;
  return 0;
}

extern "C" int dpmm_smart_set_sublabels(dpmm_ctx* ctx, int64_t cluster) {
  NEED(ctx, DPMM_EINVAL, "ctx is NULL");
  SmartState* s = ctx->smart;
  NEED(s && s->cluster >= 0 && s->cluster == (int)cluster - 1, DPMM_ESTATE, "dpmm_smart_set_sublabels: not the projected cluster");
  NEED(s->assigned, DPMM_ESTATE, "dpmm_smart_set_sublabels needs a preceding dpmm_smart_kmeans_iter");
  NEED(ctx->sorted, DPMM_ESTATE, "labels changed since dpmm_smart_project");
  CK(cudaSetDevice(ctx->device));
  if (s->cnt > 0) {
    KernelTimer kt(ctx, TK_RELABEL);
    smart_set_kernel<<<smart_grid(s->cnt), SMART_THREADS, 0, ctx->stream>>>(ctx->perm, s->beg, s->cnt, s->lab, ctx->sub);
    CK(cudaGetLastError());
  }
  ctx->partitioned = ctx->stats_cached = false;
  return 0;
}
