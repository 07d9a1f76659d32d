/*
 * dks.h -- C ABI of the B200-native KernelSHAP engine (libdks.so).
 *
 * The reference (alexcoca/DistributedKernelShap) has no FFI: its hot path is reached through a Python
 * duck-typed slot, `KernelShap._explainer` (explainers/kernel_shap.py:774-788), whose object must offer
 * `get_explanation(X, **kw)`, `.expected_value`, `.vector_out` (kernel_shap.py:789-790, :880-887).  The
 * object the reference puts there is `KernelExplainerWrapper` (kernel_shap.py:217-261), a subclass of
 * `shap.KernelExplainer` (shap==0.35.0, not vendored).  Each entry point below replaces one piece of
 * that object; the Python binding a maintainer adds is in INTEGRATION.md.
 *
 * Conventions: every function returns 0 on success or a DKS_ERR_* code; dks_last_error() returns the
 * message of the calling thread's last failure.  Plain pointers and sizes only -- no torch types.  A ctx
 * is bound to one CUDA device, owns only its workspace, and is not thread-safe.  `*_dev` pointers are
 * device memory owned by the caller (e.g. torch tensors); `*_host` pointers are host memory.  Work is
 * enqueued on the ctx stream (dks_set_stream) and is asynchronous unless the function says it
 * synchronises.  float64 at the boundary, like the reference.
 */
#ifndef DKS_H_
#define DKS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DKS_VERSION 100

/* error codes */
#define DKS_OK 0
#define DKS_ERR_INVALID 1       /* bad argument / call order */
#define DKS_ERR_CUDA 2          /* a CUDA runtime call failed (message has the CUDA error string) */
#define DKS_ERR_UNSUPPORTED 3   /* valid request the engine does not implement (never a silent fallback) */
#define DKS_ERR_PLAN_MISSING 4  /* an instance needs a coalition plan for an M that was not provided */
#define DKS_ERR_NUMERIC 5       /* normal matrix not positive definite */

/* model head applied to the linear scores z = W x + b   (replaces the opaque `predictor` callable,
 * benchmarks/ray_pool.py:34; sklearn LogisticRegression.predict_proba per scripts/fit_adult_model.py:27) */
#define DKS_ACT_IDENTITY 0      /* outputs = z (R outputs): regression / decision_function           */
#define DKS_ACT_BINARY_LOGISTIC 1 /* R = 1, outputs [1 - s, s], s = sigmoid(kappa * z): kappa = 1 is the
                                   * binary sigmoid, kappa = 2 the 2-class multinomial softmax([-z, z]) */
#define DKS_ACT_SOFTMAX 2       /* R = C >= 2 scores, outputs softmax(z)                              */

/* link (shap.common.convert_to_link; reference call sites kernel_shap.py:775, :949) */
#define DKS_LINK_IDENTITY 0
#define DKS_LINK_LOGIT 1

/* which fused kernel evaluates the coalitions (on a context set up with dks_set_mlp_model: see there) */
#define DKS_KERNEL_AUTO 0
#define DKS_KERNEL_SIMT 1       /* CUDA-core kernel (all shapes) */
#define DKS_KERNEL_TCGEN05 2    /* tensor-core kernel: Z tile x background tile on tcgen05/TMEM */
#define DKS_KERNEL_SHARED 3     /* shared-plan fast path for instances whose groups all vary (+ best general kernel
                                 * for the rest); DKS_KERNEL_AUTO picks it whenever it applies */

typedef struct dks_ctx dks_ctx;

int dks_version(void);
const char* dks_last_error(void);
/* number of CUDA devices visible to the process (0 when there is none; never an error) */
int dks_device_count(int* count);

/* ---- lifetime ------------------------------------------------------------------------------------
 * replaces KernelExplainerWrapper.__init__ (kernel_shap.py:225-229): one ctx per actor/GPU. */
int dks_create(dks_ctx** out, int device);
int dks_destroy(dks_ctx* ctx);
/* `stream` is a cudaStream_t (0 = legacy default stream).  The ctx creates its own stream by default. */
int dks_set_stream(dks_ctx* ctx, void* stream);
int dks_synchronize(dks_ctx* ctx);

/* ---- fit: shap.common.DenseData + KernelExplainer.__init__ (reached from kernel_shap.py:229) --------
 * background [N x D] row-major float64, optional weights [N] (NULL = uniform; normalised to sum 1). */
int dks_set_background(dks_ctx* ctx, const double* bg_host, int N, int D, const double* weights_host);
/* feature groups in CSR form: group g owns columns group_cols[group_offsets[g] .. group_offsets[g+1]).
 * Every column must belong to exactly one group (DenseData asserts the sizes add up to D). */
int dks_set_groups(dks_ctx* ctx, const int32_t* group_offsets, const int32_t* group_cols, int G);
/* linear scores z = W x + b with W [R x D] row-major, b [R]; head per DKS_ACT_*; kappa used by
 * DKS_ACT_BINARY_LOGISTIC only.  scalar_out != 0 marks a predictor returning a 1-D array (vector_out False). */
int dks_set_model(dks_ctx* ctx, const double* W_host, const double* b_host, int R, int activation, double kappa,
                  int scalar_out);
/* instead of dks_set_model: a network of one hidden layer of H ReLU units (scikit-learn MLPClassifier / MLPRegressor with
 * activation='relu'), scores z = W2 relu(W1 x + b1) + b2 with W1 [H x D] and W2 [R x H] row-major, b1 [H], b2 [R]; the head
 * (activation, kappa, scalar_out) as in dks_set_model.  H <= 128, R <= 8; at most 64 groups (DKS_ERR_UNSUPPORTED beyond).
 * Kernels on such a context: DKS_KERNEL_AUTO = shared-plan MLP kernel for the instances whose groups all vary (binary head,
 * uniform background weights, plans of the engine) and the general MLP kernel for the rest; DKS_KERNEL_SHARED the same, but
 * DKS_ERR_UNSUPPORTED where the shared-plan kernel does not apply; DKS_KERNEL_SIMT the general MLP kernel for every instance;
 * DKS_KERNEL_TCGEN05 is unsupported. */
int dks_set_mlp_model(dks_ctx* ctx, const double* W1_host, const double* b1_host, int H, const double* W2_host,
                      const double* b2_host, int R, int activation, double kappa, int scalar_out);
int dks_set_link(dks_ctx* ctx, int link);
/* runs the fit kernels (grouped background scores, fnull = sum_j w_j f(bg_j), link(fnull)); synchronises. */
int dks_fit(dks_ctx* ctx);
int dks_num_outputs(dks_ctx* ctx, int* C);
/* fnull[C] and expected_value[C] = link(fnull)  (KernelExplainer.fnull / .expected_value) */
int dks_get_fnull(dks_ctx* ctx, double* fnull_host, double* expected_value_host);
/* model outputs f(X) [n x C] for host rows (used to check the extracted model against the callable). */
int dks_predict_host(dks_ctx* ctx, const double* X_host, int n, double* out_host);

/* ---- coalition plans: the enumeration/sampling part of KernelExplainer.explain ----------------------
 * nsamples request shared by all instances: 0 = 'auto' (2M + 2048); capped per instance at 2^M - 2 (M<=30). */
int dks_set_nsamples(dks_ctx* ctx, int nsamples);
/* S an instance with M varying groups evaluates under the current request (upstream rule). */
int dks_effective_nsamples(dks_ctx* ctx, int M, int* S);
/* one plan shared by every instance with M varying groups: zbits [S][W] little-endian 64-bit words, W = 1 for M <= 64,
 * 2 for 64 < M <= 128 and 16 for 128 < M <= 1024 (bit k = k-th varying group present; multi-word rows are evaluated by the
 * shared-plan path only), w [S] kernel weights, in upstream row order.  Copies to the device and, up to 128 groups,
 * factors the normal matrix there. */
int dks_set_shared_plan(dks_ctx* ctx, int M, int S, const uint64_t* zbits_host, const double* w_host);
/* plans of more than 128 groups: the solve of KernelExplainer.solve (reached from kernel_shap.py:250/253; ungrouped wide
 * arrays: kernel_shap.py:581-621) in projection form, beta = P y - delta d with P = inv(E^T W E) E^T W and d = P z_L, factored
 * by the host in float64 (np.linalg.inv like upstream).  pt_host = P^T [S][M-1] row-major, dvec_host = d [M-1].  Call after
 * dks_set_shared_plan of the same M; the plan is reported present (dks_has_shared_plan) only with its projection. */
int dks_set_plan_projection(dks_ctx* ctx, int M, const double* pt_host, const double* dvec_host);
int dks_clear_plans(dks_ctx* ctx);
int dks_has_shared_plan(dks_ctx* ctx, int M, int* present);

/* ---- l1 feature selection: the l1_reg branch of KernelExplainer.solve (kwargs path kernel_shap.py:836-845, :880) --------
 * mode 0 = off (plain constrained WLS), 1 = LassoLarsIC 'aic' (what l1_reg='auto' means when under 20% of the coalition
 * space is sampled), 2 = 'bic', 3 = 'num_features(k)' (lars_path with max_iter = k); scikit-learn 0.23.2 semantics (the
 * reference's pin).  Runs on the shared-plan path for instances whose groups all vary; others_plain != 0 lets the remaining
 * instances take the plain WLS (the caller has checked that upstream would not select features for them), 0 reports them
 * as DKS_ERR_UNSUPPORTED.  dks_set_l1_tables uploads what plan.py:l1_tables computes for the shared plan of M groups (after
 * dks_set_shared_plan): Gram matrices of the augmented system [M x M], column sums / norms / b-weighted column sums [M], the
 * w-weighted Gram of the plain rows [M x M], per-row b_s and sqrt(a_s) + sqrt(b_s) [S], and three scalars. */
int dks_set_l1(dks_ctx* ctx, int mode, int k, int others_plain);
int dks_set_l1_tables(dks_ctx* ctx, int M, const double* gram_raw, const double* gram_norm, const double* colsum,
                      const double* scale, const double* bz, const double* gram_w, const double* b_rows,
                      const double* sqab_rows, double sum_b, double sum_sqb, int n_aug);

/* ---- per-instance plans drawn on the device -----------------------------------------------------------
 * shap.KernelExplainer.explain draws a fresh plan for every instance (the sampling loop that follows the subset
 * enumeration; reached from kernel_shap.py:250/253).  Mode 1 does that on the GPU: the enumerated prefix comes from the
 * shared plan of the instance's M, the sampled rows from Philox4x32-10 keyed by `seed` with counter (draw, global row),
 * with upstream's duplicate / complement / truncation / rescaling rules.  Plans depend on the global row index only
 * (dks_set_row_offset gives the index of row 0 of the next call), never on batching or the number of GPUs.
 * dks_set_plan_sampling uploads what the sampler needs for one M (plan.py: sampling_info); cdf has ncdf <= 32 entries. */
int dks_set_plan_sampling(dks_ctx* ctx, int M, int nfixed, int n_full, int n_paired, int ncdf, const double* cdf_host,
                          double weight_left);
int dks_set_plan_mode(dks_ctx* ctx, int mode /* 0 shared per M, 1 per instance */, uint64_t seed);
int dks_set_row_offset(dks_ctx* ctx, int64_t offset);
/* plans of the last mode-1 explain call ([n][stride] each; pass NULL buffers to query n and stride); tests / audit. */
int dks_get_instance_plans(dks_ctx* ctx, uint64_t* zbits_host, double* w_host, int* n_out, int* stride_out);

/* ---- explain: KernelExplainer.shap_values (reached from kernel_shap.py:250/253) ---------------------
 * Stage 1 (dks_prepare_*): per instance, grouped contributions W_g x_g, f(x), link(f(x)) - link(fnull),
 * varying_groups() bit-mask and M.  X is [n x D] row-major float64. */
int dks_prepare_host(dks_ctx* ctx, const double* X_host, int n);
int dks_prepare_dev(dks_ctx* ctx, const double* X_dev, int n);
/* after prepare: hist[m] = number of instances with M == m, m in [0, G]; synchronises. */
int dks_get_m_histogram(dks_ctx* ctx, int32_t* hist_host);
/* after prepare / explain: link(f(x)) per instance and output, [n][C] -- what KernelShap.build_explanation stores as
 * `raw_prediction` (kernel_shap.py:949 runs the predictor over X a second time for it); synchronises. */
int dks_get_link_fx(dks_ctx* ctx, double* out_host, int n /* rows the caller's buffer holds: must match */);
/* after prepare: per-instance M and varying bit-mask (debug / tests); synchronises. */
int dks_get_varying(dks_ctx* ctx, int32_t* M_host, uint64_t* mask_host);

/* Stage 2: evaluate coalitions + solve.  phi is [C x n x G] float64 (one [n x G] slab per model output,
 * the list-of-arrays layout KernelExplainer.shap_values returns).
 * Plans: ext_zbits/ext_w == NULL -> shared plans (dks_set_shared_plan) looked up by each instance's M;
 * otherwise per-instance plans [n x ext_stride] (row i holds the S_i = dks_effective_nsamples(M_i) rows of
 * instance i), device pointers for _dev and host pointers for _host. */
int dks_explain_dev(dks_ctx* ctx, double* phi_dev, const uint64_t* ext_zbits_dev, const double* ext_w_dev,
                    int ext_stride);
/* prepare + explain for rows resident in device memory with the engine's own plans, as ONE CUDA-graph launch once the
 * same call (same buffers, n, nsamples, kernel, plans) has been seen twice: the second call captures the sequence (memset,
 * stage 1, coalition kernels, solve), later ones replay it.  DKS_GRAPH=0 in the environment keeps plain launches.
 * Asynchronous like dks_explain_dev; dks_last_timings keeps working (external event-record nodes). */
int dks_run_dev(dks_ctx* ctx, const double* X_dev, int n, double* phi_dev);
int dks_graph_launches(dks_ctx* ctx, int64_t* count);
/* Multi-GPU, one process per GPU: gathered_ptrs_host[r] is the device address, valid in THIS process (peer mapping, e.g.
 * torch symmetric memory), of rank r's gathered buffer [world][slab_doubles].  After every dks_run_dev the engine stores
 * its phi into slab `rank` of every peer's buffer with its own kernel over NVLink peer memory -- the all-gather of the
 * reference's result collection (distributed.py:156-179) without NCCL; the caller completes it with a cross-GPU barrier.
 * Pass phi_dev = own buffer + rank * slab_doubles to have the solve write the local slab in place.  world <= 1 clears. */
int dks_set_peers(dks_ctx* ctx, int world, int rank, const uint64_t* gathered_ptrs_host, int64_t slab_doubles);
/* Optional completion of that all-gather inside the engine: flag_ptrs_host[r] is the device address (mapped in THIS process) of
 * rank r's flag array, uint64[world], zero-initialised (peer-mapped like the gathered buffers).  With flags set, every
 * dks_run_dev ends with the engine's own cross-GPU signal/wait (one thread per peer, system-scope release/acquire): when the
 * call's stream work is done, every peer's block has arrived in this rank's gathered buffer -- no library barrier needed.
 * Call after dks_set_peers; NULL switches it off. */
int dks_set_peer_flags(dks_ctx* ctx, const uint64_t* flag_ptrs_host);
/* convenience: prepare + explain from/to host memory; H2D, kernels, D2H; synchronises.  This is the call a
 * non-torch host (ctypes / cgo) makes and the one bench.py's end-to-end number goes through. */
int dks_explain_host(dks_ctx* ctx, const double* X_host, int n, double* phi_host, const uint64_t* ext_zbits_host,
                     const double* ext_w_host, int ext_stride);
/* Page-locked host memory for result arrays (optional).  When the phi_host handed to dks_explain_host lies in page-locked
 * memory (allocated here, or registered by the caller) the shap values arrive by ONE asynchronous DMA; pageable memory goes
 * through the library's pinned staging buffer and a host memcpy. */
int dks_host_alloc(void** out, uint64_t bytes);
int dks_host_free(void* p);
/* status of the LAST explain call on this context (the asynchronous calls leave it on the device; this fetches it and
 * synchronises): 0 ok, DKS_ERR_PLAN_MISSING, DKS_ERR_NUMERIC, DKS_ERR_UNSUPPORTED;
 * *detail = the offending M / instance index. */
int dks_last_status(dks_ctx* ctx, int* detail);

/* ---- post-processing of KernelShap.build_explanation off the resident phi (kernel_shap.py:36-109 rank_by_importance, :112-207
 * sum_categories, :952-956 argmax) for the rows of the LAST dks_explain_host call: segment sums over consecutive groups
 * (seg_offsets_host [Gp + 1], NULL = one segment per group, Gp = G), mean |phi| per output and aggregated over outputs
 * ([C + 1][Gp]), their descending order, argmax of the raw prediction.  Output pointers may be NULL.  Synchronises. */
int dks_summarise_host(dks_ctx* ctx, int n, const int32_t* seg_offsets_host, int Gp, double* phi_sum_host,
                       double* mean_abs_host, int32_t* order_host, int32_t* argmax_host);

/* ---- knobs / introspection ---------------------------------------------------------------------- */
int dks_set_kernel(dks_ctx* ctx, int kernel);       /* DKS_KERNEL_* */
/* tuning knobs, all optional (defaults are the measured best): "fused" 0/1 -- link + projection solve inside the shared-plan
 * coalition kernel (default 1; 0 = separate (sum p1, sum p0) buffer + solve kernel); "fused_ni" 1/2 instances per pass over
 * a warp's rows; "fused_warps" 16/20 warps per CTA; "fused_batch" instances parked per warp before the turn-around;
 * "push_in_kernel" 0/1 -- multi-GPU: the fused kernel's epilogue stores phi into the peers' buffers itself instead of the
 * separate push kernel (default 0: measured slower, it stalls the finishing warps); "graph" 0/1 (CUDA-graph
 * replay of dks_run_dev); "graph_timing" 0/1 -- keep the timing event records inside the graph (default 0: a replayed graph
 * carries no timing nodes and dks_last_timings reports an error after it); plans of more than 128 groups: "wide_gemm" 1/2 --
 * float64 product of the projection solve, 2 = 128 x 64 tiles with conflict-free 128-bit shared-memory operands (default),
 * 1 = the first 64 x 64 version; "wide_acache" 0/1 -- A(i, s) of sixteen-word rows computed by the first background
 * chunk's launch only (default 1).  Both give identical bits either way. */
int dks_set_option(dks_ctx* ctx, const char* name, int value);
int dks_kernel_launches(dks_ctx* ctx, int64_t* count); /* kernels launched by this ctx so far */
/* device-time of the last explain's stages in ms (CUDA events on the ctx stream): [0] prepare, [1] fused
 * coalition kernel, [2] total; synchronises. */
int dks_last_timings(dks_ctx* ctx, float* ms3);

/* ---- debugging aid for the tcgen05 kernel (tests only) ---------------------------------------------------
 * dks_debug_score_dump(ctx, i): the next explains also write the raw accumulator tile of instance i (scaled masked
 * scores T[s][j], float32 [rows x cols]); i < 0 switches it off.  dks_debug_get_scores copies the dump to the host
 * (synchronises); rows/cols report its shape. */
int dks_debug_score_dump(dks_ctx* ctx, int instance);
int dks_debug_get_scores(dks_ctx* ctx, float* out_host, int max_floats, int* rows, int* cols);
/* cycle timeline of CTA 0 recorded by the same debug run: float32 [6][256], event e of tile g at [e*256+g]
 * (0 A-tile ready, 1 accumulator free, 2 MMAs issued, 3 epilogue waits, 4 accumulator full, 5 accumulator drained) */
int dks_debug_get_timeline(dks_ctx* ctx, float* out_host);

#ifdef __cplusplus
}
#endif
#endif /* DKS_H_ */
