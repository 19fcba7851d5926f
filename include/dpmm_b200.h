/*
 * dpmm_b200.h -- C ABI of libdpmm_b200.so: the B200 (sm_100a) data-parallel sweep of the
 * DPMM sub-cluster sampler.
 *
 * This library replaces the WORKER side of DPMMSubClusters.jl (v0.1.13): everything the master
 * reaches through Distributed.@spawnat / remotecall in src/local_clusters_actions.jl.  The host
 * (Julia, or the Python mirror shipped in this repo) keeps fit()/dp_parallel(), the prior plugin
 * types, calc_posterior, parameter sampling and the Hastings ratios.  Every entry point below names
 * the reference call site it replaces (file:line under the reference tree).
 *
 * Conventions
 *   - plain C, no exceptions; every call returns 0 on success or a negative DPMM_E* code, and
 *     dpmm_last_error(ctx) returns a human-readable message (ctx may be NULL for create failures).
 *   - one context = one GPU = one shard of the points (one "worker" of the reference); one host
 *     thread per context; calls are enqueued on the context's CUDA stream in call order (the
 *     reference relies on per-worker FIFO order of @spawnat tasks, local_clusters_actions.jl:64-68,
 *     102-109 -- a stream gives the same semantics).  Calls that return data synchronise.
 *   - labels and sub-labels cross the boundary as 1-based int64 (Julia Int64, ds.jl:54-55);
 *     cluster indices in index lists are 1-based int64 as well.
 *   - points are float32, D x N column-major (each point = D contiguous floats, ds.jl:53), or, for the
 *     multinomial prior, sparse compressed columns (dpmm_create_sparse).
 *   - host buffers are borrowed for the duration of the call only (x is copied at create).
 *   - there is NO CPU fallback: without a CUDA device every call fails with DPMM_ECUDA.
 */
#ifndef DPMM_B200_H
#define DPMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPMM_OK 0
#define DPMM_EINVAL (-1)   /* bad argument                                   */
#define DPMM_ECUDA (-2)    /* CUDA runtime error / no device                 */
#define DPMM_ESTATE (-3)   /* call order violated (e.g. sampling before set_params) */
#define DPMM_ELIMIT (-4)   /* size outside the supported range (see dpmm_limits)    */
#define DPMM_ENCCL (-5)    /* NCCL error                                      */

#define DPMM_PRIOR_NIW 0          /* niw_hyperparams   -> mv_gaussian       (src/priors/niw.jl)               */
#define DPMM_PRIOR_MULTINOMIAL 1  /* multinomial_hyper -> multinomial_dist  (src/priors/multinomial_prior.jl) */
#define DPMM_PRIOR_DIAG_GAUSSIAN 2 /* diag_niw_hyperparams -> diag_gaussian: an independent D = 1 NIW per feature   */

#define DPMM_SAMPLER_INVERSE_CDF 0 /* reference semantics: StatsBase.sample(ProbabilityWeights), utils.jl:29 */
#define DPMM_SAMPLER_GUMBEL 1      /* Gumbel-max: same distribution, different stream, no per-point K storage */

typedef struct dpmm_ctx dpmm_ctx;

/* ---- lifetime ------------------------------------------------------------------------------ */

/* init_model_from_data: `data = distribute(all_data)` (src/dp-parallel-sampling.jl:42-44) for ONE
 * shard.  x: host float32 [d x n_local] column-major, copied to the device.  global_offset = index
 * (0-based) of this shard's first point in the whole data set: the counter-based RNG is keyed by the
 * global point index so results do not depend on how many GPUs the points are spread over.
 * device: CUDA ordinal.  seed: replaces `@everywhere Random.seed!(seed)` (:37-39).
 * d: 1..64 for the NIW prior, 1..16384 for the multinomial and the diagonal Gaussian prior; larger d returns
 * DPMM_ELIMIT.  Every multinomial or diagonal d samples with any K up to DPMM_MAX_K.  A diagonal Gaussian context
 * runs the sweep and, after dpmm_set_hyper_diag, the device parameter step; dpmm_predict_* and dpmm_smart_* return
 * DPMM_ESTATE on it. */
int dpmm_create(dpmm_ctx** out, const float* x, int64_t n_local, int32_t d, int32_t prior_kind,
                int32_t device, uint64_t seed, int64_t global_offset);
/* init_model_from_data for ONE shard of sparse counts: the three arrays of a Julia SparseMatrixCSC{Float32,Int64}
 * of size d x n_local (column j = point j), 1-based as Julia stores them.  Multinomial prior only.
 *   colptr int64 [n_local + 1]  colptr[0] == 1, non-decreasing; nnz = colptr[n_local] - 1 >= 0
 *   rowval int64 [nnz]          1..d, strictly increasing within a column
 *   nzval  float32 [nnz]
 * Empty columns and nnz = 0 are valid.  n_local, d, colptr[0] and nnz are checked on the host (d > 16384:
 * DPMM_ELIMIT); the arrays are then copied to the device and checked there while they are converted to the internal
 * layout (compressed rows: int64 offsets, int32 feature indices, float32 counts): a violation returns DPMM_EINVAL
 * naming the first invalid column.  global_offset, device and seed as for dpmm_create.
 * A sparse context has every entry point of a dense multinomial context holding the same matrix except the smart-split
 * projection (dpmm_smart_project: DPMM_ESTATE).  Its log-likelihoods are the sequential Float32 fmaf chain over the
 * stored entries in ascending feature order: bit for bit what the dense kernels compute over all D features, with
 * one deliberate difference: a -Inf log-probability against a zero count (stored or not) contributes nothing, where
 * the dense product gives NaN (0 * -Inf).  That is also what Julia's sparse `alpha' * x` gives for absent entries. */
int dpmm_create_sparse(dpmm_ctx** out, const int64_t* colptr, const int64_t* rowval, const float* nzval,
                       int64_t n_local, int32_t d, int32_t device, uint64_t seed, int64_t global_offset);
int dpmm_destroy(dpmm_ctx* ctx);
const char* dpmm_last_error(const dpmm_ctx* ctx);
/* Use an externally owned cudaStream_t (e.g. the host framework's current stream) for all work. */
int dpmm_set_stream(dpmm_ctx* ctx, void* cuda_stream);
int dpmm_sync(dpmm_ctx* ctx);
/* out[0]=max D (NIW, 64), out[1]=max D (multinomial and diagonal Gaussian, 16384), out[2]=max K (1024, any D of
 * every prior). */
int dpmm_limits(int32_t* out3);

/* ---- labels: initialisation, gather, resume ------------------------------------------------- */

/* labels = rand(1:init_clusters, N) (+1 if outlier); sub-labels = rand(1:2, N)
 * (src/dp-parallel-sampling.jl:49-50). */
int dpmm_init_labels(dpmm_ctx* ctx, int32_t init_clusters, int32_t outlier);
/* split_first_cluster_worker! (local_clusters_actions.jl:257-261) when indices==NULL: all
 * sub-labels <- rand(1:2); reset_bad_clusters_worker! / rand_subclusters_labels! (:474-488)
 * otherwise: only points whose label is listed. */
int dpmm_randomize_sublabels(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices);
/* Array(group.labels) / Array(group.labels_subcluster) (dp-parallel-sampling.jl:218,276,371;
 * ds.jl:85-87).  out: host int64[n_local]. */
int dpmm_get_labels(dpmm_ctx* ctx, int64_t* out);
int dpmm_get_sublabels(dpmm_ctx* ctx, int64_t* out);
/* distribute(group.labels) on resume (dp-parallel-sampling.jl:437-438). */
int dpmm_set_labels(dpmm_ctx* ctx, const int64_t* labels);
int dpmm_set_sublabels(dpmm_ctx* ctx, const int64_t* sublabels);

/* ---- parameters ------------------------------------------------------------------------------ */

/* broadcast_cluster_params -> set_global_data (local_clusters_actions.jl:518-549): ship the thin
 * cluster parameters (ds.jl:29-34) and the mixture weights.  Distributions are ordered
 * [cluster k][cluster_dist, l_dist, r_dist], i.e. 3*K of them.
 *   mu        float32 [3K][D]        mv_gaussian.mu        (mv_gaussian.jl:13)
 *   inv_sigma float32 [3K][D][D]     mv_gaussian.invSigma  (:15; symmetric, either major order)
 *   logdet    float32 [3K]           mv_gaussian.logdetSigma (:16)
 *   weights   float32 [K]            group.weights (ds.jl:57);  lr_weights float32 [K][2] (ds.jl:33)
 * The library factors invSigma = U'U on the device in float64 (niw_pack_kernel; the reference carries
 * the same factor in mv_gaussian.invChol, :17) and evaluates z'invSigma z as |U z|^2. */
int dpmm_set_params_niw(dpmm_ctx* ctx, int32_t k, const float* mu, const float* inv_sigma,
                        const float* logdet, const float* weights, const float* lr_weights);
/* log_p float32 [3K][D] = multinomial_dist.alpha (log-probabilities, multinomial_dist.jl:8-10). */
int dpmm_set_params_multinomial(dpmm_ctx* ctx, int32_t k, const float* log_p, const float* weights,
                                const float* lr_weights);
/* Diagonal Gaussian distributions (diag_gaussian), same order and weights as dpmm_set_params_niw:
 *   mu float32 [3K][D], var float32 [3K][D] (sigma^2_d > 0), logdet float32 [3K] (sum_d log sigma^2_d).
 * The log-likelihood is -(D log 2pi + logdet)/2 - 1/2 sum_d ((x_d - mu_d)/sigma_d)^2 in Float32, evaluated as
 * t = fma(s_d, x_d, -s_d mu_d) with s_d = 1/sigma_d (rounded once from Float64), then sum t^2.  The images are
 * derived on the device by the same kernel that packs device-sampled parameters (dpmm_sample_params), so that
 * dpmm_get_params_diag -> dpmm_set_params_diag reproduces them bit for bit. */
int dpmm_set_params_diag(dpmm_ctx* ctx, int32_t k, const float* mu, const float* var, const float* logdet,
                         const float* weights, const float* lr_weights);
int dpmm_set_sampler(dpmm_ctx* ctx, int32_t sampler);

/* ---- the sweep ------------------------------------------------------------------------------- */

/* sample_labels! -> sample_labels_worker! (local_clusters_actions.jl:98-134): per point
 * log-likelihood under every cluster_dist + log weight, then (final != 0) first-argmax or
 * sample_log_cat_array! (utils.jl:19-31).  The N x K matrix is never written to memory. */
int dpmm_sample_labels(dpmm_ctx* ctx, int32_t final_iter);
/* sample_sub_clusters! -> sample_sub_clusters_worker! -> create_subclusters_labels! (:64-95):
 * each point, under the l/r distributions of its (fresh) label.  For NIW models with D = 32 the same
 * kernel also accumulates the left/right statistics of every cluster; a dpmm_suff_stats call that
 * follows without a label / sub-label change in between is served from them. */
int dpmm_sample_sublabels(dpmm_ctx* ctx);
/* update_suff_stats_posterior! -> create_suff_stats_dict_worker (:149-169, :206-254) with
 * create_sufficient_statistics (niw.jl:42-51, multinomial_prior.jl:27-32) and the worker->leader->
 * master aggregate_suff_stats reduction (niw.jl:64-66, :171-203, :246-248), which becomes one NCCL
 * all-reduce when a communicator is attached.
 * indices: 1-based cluster indices (NULL = all K clusters, n_indices ignored).  Outputs (host, may
 * each be NULL; if all are NULL the statistics are left on the device and the call does not
 * synchronise), m = number of indices:
 *   counts  int64  [m][3]            N of {cluster, left, right}
 *   sum_x   double [m][3][D]         points_sum
 *   sum_xx  double [m][3][D][D]      S (symmetric; NIW),  double [m][3][D]  sum of x_d^2 per feature (diagonal
 *                                    Gaussian); ignored for multinomial
 * Gaussian statistics are accumulated in Float64. */
int dpmm_suff_stats(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices, int64_t* counts,
                    double* sum_x, double* sum_xx);

/* Number of label values in use = max(K of the last set_params, largest label): the row count of a
 * dpmm_suff_stats(indices = NULL) result.  With indices == NULL, n_indices must be 0 or exactly this. */
int dpmm_num_clusters(const dpmm_ctx* ctx);

/* ---- device-side parameter step (NIW and multinomial; SURVEY 8f-1) ----------------------------
 * Optional: the host may keep sampling parameters itself (dpmm_set_params_*).  With these calls the
 * per-iteration master work that scales with K D^3 (NIW) or K D (multinomial, diagonal Gaussian) runs next to the
 * statistics:
 *   calc_posterior / log_marginal_likelihood   src/priors/niw.jl:20-31, 53-62; multinomial_prior.jl:16-21, 34-39
 *   sample_distribution                        src/priors/niw.jl:34-40; multinomial_prior.jl:23-25
 *   sample_cluster_params / sample_clusters!   src/shared_actions.jl:41-66, src/local_clusters_actions.jl:417-437
 *   should_merge! (the merged log marginal)    src/shared_actions.jl:21-38
 * The host keeps the Hastings accept / reject decisions on 3K scalars (+ the K x K merge table).
 * Every D below is the caller's d of dpmm_create, also where the NIW context runs zero-padded to a wider kernel. */

/* niw_hyperparams (niw.jl:6-11: kappa, m[D], nu, psi[D][D]) and the concentration alpha (ds.jl:9).
 * DPMM_EINVAL unless kappa > 0, nu > D - 1, alpha > 0 and psi is positive definite. */
int dpmm_set_hyper_niw(dpmm_ctx* ctx, double kappa, const double* m, double nu, const double* psi, double alpha);
/* multinomial_hyper (multinomial_prior.jl:6-8: alpha_prior float32 [D], every entry finite and > 0) and the
 * concentration alpha > 0 (ds.jl:9).  DPMM_ESTATE on an NIW context. */
int dpmm_set_hyper_multinomial(dpmm_ctx* ctx, const float* alpha_prior, double alpha);
/* diag_niw_hyperparams (kappa, m double [D], nu, psi double [D]: an independent NIW at D = 1 per feature, shared kappa
 * and nu) and the concentration alpha.  kappa, nu and alpha are kept rounded to Float32.  DPMM_EINVAL for a NULL
 * pointer, kappa <= 0, nu <= 0, alpha <= 0, a non-finite m[d] or a psi[d] that is not finite and > 0; DPMM_ESTATE on
 * a context of another prior. */
int dpmm_set_hyper_diag(dpmm_ctx* ctx, double kappa, const double* m, double nu, const double* psi, double alpha);
/* The outlier component (DESIGN.md 6.1): cluster 1 becomes a cluster under a prior of its own with the fixed mixture
 * weight fl32(weight); the other weights are (1 - weight) Dirichlet(N_2..N_K, alpha), or (1 - weight) / (K - 1) with
 * unit_weights.  The posterior, draws (from_prior too) and log marginal likelihood of cluster 1 use this prior; the
 * sweep is unchanged.  The host never splits or merges cluster 1 (dpmm_params_merge refuses it) and keeps it through
 * dpmm_remove_empty.  Each call follows the matching dpmm_set_hyper_* (DPMM_ESTATE before it or on a context of another
 * prior), validates the prior exactly as dpmm_set_hyper_* does and needs 0 <= weight < 1 (DPMM_EINVAL otherwise);
 * weight = 0 turns the component off again. */
int dpmm_set_outlier_niw(dpmm_ctx* ctx, double weight, double kappa, const double* m, double nu, const double* psi);
int dpmm_set_outlier_multinomial(dpmm_ctx* ctx, double weight, const float* alpha_prior);
int dpmm_set_outlier_diag(dpmm_ctx* ctx, double weight, double kappa, const double* m, double nu, const double* psi);
/* update_suff_stats_posterior! (local_clusters_actions.jl:206-254) kept on the device: statistics of the
 * listed clusters (NULL = all) -> all-reduce -> persistent table -> posterior hyper-parameters and log
 * marginal likelihoods of {cluster, left, right}.  from_table != 0: skip the statistics and re-evaluate the
 * listed table rows (after dpmm_params_merge).  splittable[k_merge] (optional): also evaluate, for every
 * pair i < j of splittable non-empty clusters, the log marginal likelihood of the merged cluster
 * (check_and_merge!, :385-413) into merge_logml[k_merge][k_merge] (NaN elsewhere).
 * Outputs (host, optional): counts int64 [m][3], logml double [m][3].  Synchronises iff an output is given. */
int dpmm_posterior_step(dpmm_ctx* ctx, const int64_t* indices, int32_t n_indices, int32_t from_table,
                        const uint8_t* splittable, int32_t k_merge, int64_t* counts, double* logml,
                        double* merge_logml);
/* sample_clusters! + broadcast_cluster_params (:417-437, :518-549) on the device: draw the 3K distributions
 * from the posterior table (from_prior != 0: from the prior), the sub-cluster weights Dirichlet(N_l + a/2,
 * N_r + a/2) and the mixture weights Dirichlet(N_1..N_K, a) (unit_weights != 0: 1/K, as
 * init_first_clusters!, dp-parallel-sampling.jl:77), and pack them for the sweep.  Replaces dpmm_set_params_*. */
int dpmm_sample_params(dpmm_ctx* ctx, int32_t k, int32_t from_prior, int32_t unit_weights);
/* merge_clusters_to_splittable (shared_actions.jl:12-18) on the statistics table: cluster i <- {i + j, i, j},
 * cluster j <- empty (1-based).  Follow with dpmm_posterior_step(from_table = 1) for i.  DPMM_EINVAL for i or j = 1
 * while the outlier component is on. */
int dpmm_params_merge(dpmm_ctx* ctx, int64_t i, int64_t j);
/* The parameters of the last dpmm_sample_params: mu float32 [3K][D], lfac double [3K][D][D] (L lower,
 * invSigma = L L'), logdet float32 [3K] (log det Sigma), weights float32 [K], lr_weights float32 [K][2]; D is the
 * caller's (the padded features of a zero-padded context are not returned). */
int dpmm_get_params_niw(dpmm_ctx* ctx, int32_t k, float* mu, double* lfac, float* logdet, float* weights,
                        float* lr_weights);
/* The parameters of the last dpmm_sample_params of a multinomial context: log_p float32 [3K][D]
 * (multinomial_dist.alpha), weights float32 [K], lr_weights float32 [K][2].  Each output may be NULL. */
int dpmm_get_params_multinomial(dpmm_ctx* ctx, int32_t k, float* log_p, float* weights, float* lr_weights);
/* The parameters of the last dpmm_sample_params of a diagonal Gaussian context (diag_gaussian): mu float32 [3K][D],
 * var float32 [3K][D] (sigma^2), logdet float32 [3K] (sum_d log sigma^2_d over the Float32 var), weights float32 [K],
 * lr_weights float32 [K][2].  Each output may be NULL.  DPMM_ESTATE without device-sampled parameters for this K. */
int dpmm_get_params_diag(dpmm_ctx* ctx, int32_t k, float* mu, float* var, float* logdet, float* weights,
                         float* lr_weights);

/* predict / predict_points (src/dp-parallel-sampling.jl:509-537, src/local_clusters_actions.jl:23-40) for the
 * points of THIS context under K NIW posterior predictives (multivariate Student-t, niw.jl:68-76):
 *   parr[i,k] = tconst[k] - (df[k] + D)/2 * log1p(|U_k (x_i - mu_k)|^2 / df[k])
 * u float32 [K][D][D] = rows of the upper factor of the inverse scale matrix, tconst = the density's constant
 * plus log weight (the host prepares both from the K posterior hyper-parameters).  labels: int64 [n] (1-based
 * first argmax); probs: float32 [n][K] softmax over k, or NULL. */
int dpmm_predict_niw(dpmm_ctx* ctx, int32_t k, const float* u, const float* mu, const float* tconst,
                     const float* df, int64_t* labels, float* probs);
/* The same for K multinomial posterior predictives (multinomial_prior.jl:45-48):
 *   parr[i,k] = fl32(logp_k' x_i) + logw[k]   (dot product in float64, the sum in float32)
 * logp double [K][D] = log(alpha'_k / sum alpha'_k), logw float32 [K] = log of the mixture weights.  labels: int64 [n]
 * (1-based first argmax, NaN counts as maximal); probs: float32 [n][K] softmax over k (NaN as -Inf), or NULL. */
int dpmm_predict_multinomial(dpmm_ctx* ctx, int32_t k, const double* logp, const float* logw, int64_t* labels,
                             float* probs);

/* ---- relabelling after split / merge / compaction ------------------------------------------- */

/* split_cluster_local_worker! (local_clusters_actions.jl:265-278). */
int dpmm_apply_split(dpmm_ctx* ctx, const int64_t* indices, const int64_t* new_indices, int32_t n);
/* merge_clusters_worker! (:293-304). */
int dpmm_apply_merge(dpmm_ctx* ctx, const int64_t* indices, const int64_t* new_indices, int32_t n);
/* remove_empty_clusters_worker! (:446-455); pts_count[k] as the host holds it. */
int dpmm_remove_empty(dpmm_ctx* ctx, const int64_t* pts_count, int32_t k);

/* ---- smart splits (SURVEY 8f-3; smart_cluster_init! src/local_clusters_actions.jl:555-623) ---- */

/* tranform_points_worker! (:641-652) for every shard + the master's reduction (:578-589): projects the points whose
 * label is `cluster` (1-based) onto v, t = v'(x - mu) in Float64 (v, mu: double [D]), keeps t on the device and
 * returns lo_hi[0] = the minimum over shards of percentile(t, 0.10), lo_hi[1] = the maximum over shards of
 * percentile(t, 0.90) (StatsBase semantics: the p/100 quantile; shards with fewer than 2 such points do not take
 * part; NaN when none does) and *count = the number of such points over all shards. */
int dpmm_smart_project(dpmm_ctx* ctx, int64_t cluster, const double* v, const double* mu, double* lo_hi,
                       int64_t* count);
/* kmeans_iter_worker! (:633-639) + the master's sums (:601-612): assigns every projected point to the nearer of
 * (min_mean, max_mean) (ties -> max_mean) and returns out4 = {sum_1, count_1, sum_2, count_2} over all shards. */
int dpmm_smart_kmeans_iter(dpmm_ctx* ctx, double min_mean, double max_mean, double* out4);
/* set_smart_labels_in_worker! (:627-631): sub-labels of the projected cluster <- the last assignment. */
int dpmm_smart_set_sublabels(dpmm_ctx* ctx, int64_t cluster);

/* ---- multi-GPU (one process per GPU) --------------------------------------------------------- */

/* 128-byte ncclUniqueId, created on rank 0 and shipped to the other ranks by the host's own means. */
int dpmm_nccl_unique_id(void* out128);
int dpmm_comm_init(dpmm_ctx* ctx, const void* unique_id128, int32_t rank, int32_t world_size);

/* ---- parity / measurement hooks -------------------------------------------------------------- */

/* Inject randomness (host arrays of length n_local, or NULL to return to Philox):
 * u_label / u_sub: the one uniform each point consumes in the label / sub-label draw;
 * r_bits: the rand(1:2)-1 bit used by randomize_sublabels / apply_split. */
int dpmm_set_uniforms(dpmm_ctx* ctx, const double* u_label, const double* u_sub, const uint8_t* r_bits);
/* which=0: out float32 [n_local x K] column-major = parr of sample_labels_worker! (:120-127);
 * which=1: out float32 [n_local x 2] = the l/r matrix of create_subclusters_labels! (:89-93) under
 * each point's current label. */
int dpmm_debug_loglik(dpmm_ctx* ctx, int32_t which, float* out);
/* Tensor-core label path diagnostics (set DPMM_TC_STATS=1): out[0] = points drawn, out[1] = exact
 * (FP32-refined) cluster evaluations of the last dpmm_sample_labels (both 0 when the FMA path ran),
 * out[2] = points of that call finished by the full-K overflow kernel (NaN screen values or more than
 * 7 candidate clusters; D = 32 / 64 path). */
int dpmm_debug_tc_stats(dpmm_ctx* ctx, int64_t* out3);
/* Label sort diagnostics: perm (n_local entries, or NULL) receives the point indices in the order of the current
 * label sort (sorting first if needed), moved[0] the number of points whose label changed in the last dpmm_sample_labels
 * that ran on the D = 32 / 64 tensor-core path (the sort after such a call skips its scatter when it is 0). */
int dpmm_debug_sort(dpmm_ctx* ctx, int32_t* perm, int64_t* moved);
/* Fused sub-label + statistics path diagnostics (NIW, D = 32): out[0] = launches of the fused kernel by
 * dpmm_sample_sublabels, out[1] = dpmm_suff_stats calls served from its accumulators, out[2] = calls that
 * fell back to the separate statistics kernel because a run lay far from its cluster's centre. */
int dpmm_debug_fused_stats(dpmm_ctx* ctx, int64_t* out3);
/* Per-kernel device timing (CUDA events around every launch) for roofline reporting. */
int dpmm_timing_enable(dpmm_ctx* ctx, int32_t on);
int dpmm_timing_kinds(void);
const char* dpmm_timing_name(int32_t kind);
/* Synchronises; ms[kind] = summed device time, launches[kind] = count since enable/reset. */
int dpmm_timing_read(dpmm_ctx* ctx, double* ms, int64_t* launches, int32_t reset);
/* Number of kernels this context has launched since creation. */
int64_t dpmm_launch_count(const dpmm_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* DPMM_B200_H */
