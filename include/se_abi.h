/*
 * se_abi.h — C ABI of libse_b200.so: the B200-native (sm_100a) row-parallel boosting hot path of
 * pierrenodet/spark-ensemble.  This is the drop-in boundary: the entry points below are what the
 * reference's Scala train()/predict() bodies bind through JNI (jni/se_jni.cpp) once their per-row
 * RDD closures are replaced by native calls; the same symbols are driven through ctypes by
 * spark_ensemble_b200/ (host-side mirror of the Spark ML surface) and by tests/.
 *
 * Reference citations are relative to /root/reference/core/src/main/scala/org/apache/spark/ml/.
 *
 * Conventions
 *  - plain C: opaque handle, int status (0 = SE_OK, negative = error; text via se_last_error()),
 *    plain pointers and sizes, no exceptions cross the boundary, no torch/CUDA types in signatures.
 *  - one se_ctx == one GPU == one row shard.  A context is single-threaded by contract (the Spark
 *    driver thread / one executor task); distinct contexts may be used concurrently.
 *  - device state is column-major fp32: per-row arrays are [dim][n_local] ("class-major", rows
 *    contiguous), model-output matrices are [M][n_local] or [M][K][n_local].  Host buffers passed to
 *    se_upload/se_download are borrowed for the duration of the call only.
 *  - every scalar result is fp64 and GLOBAL: when a communicator is attached (se_comm_init) the
 *    per-GPU partial sums are all-reduced (one NCCL allreduce of <= dim+3 doubles over NVLink) before
 *    they are returned, exactly where the reference calls treeAggregate/treeReduce.
 *  - there is no CPU fallback: every compute entry point fails with SE_ERR_CUDA if no device works.
 */
#ifndef SE_ABI_H
#define SE_ABI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SE_ABI_VERSION 1

/* exported with default visibility; everything else in the library is hidden */
#if defined(__GNUC__)
#define SE_API __attribute__((visibility("default")))
#else
#define SE_API
#endif

/* status codes */
#define SE_OK 0
#define SE_ERR_ARG (-1)    /* IllegalArgumentException on the Scala side */
#define SE_ERR_CUDA (-2)   /* RuntimeException */
#define SE_ERR_NCCL (-3)
#define SE_ERR_STATE (-4)  /* call order / missing slot */
#define SE_ERR_OPT (-5)    /* optimiser exceeded MaxEval (TooManyEvaluationsException in the reference) */

typedef struct se_ctx se_ctx;

/* ---- losses: boosting/GBMLoss.scala:129-318 ------------------------------------------------- */
enum se_loss {
  SE_LOSS_SQUARED = 0,        /* SquaredLoss :129-137 */
  SE_LOSS_ABSOLUTE = 1,       /* AbsoluteLoss :139-143 */
  SE_LOSS_HUBER = 2,          /* HuberLoss(delta) :168-177            param = delta */
  SE_LOSS_QUANTILE = 3,       /* QuantileLoss(q) :179-188             param = q */
  SE_LOSS_LOGCOSH = 4,        /* LogCoshLoss :145-152 */
  SE_LOSS_SCALED_LOGCOSH = 5, /* ScaledLogCoshLoss(alpha) :154-166    param = alpha */
  SE_LOSS_BERNOULLI = 6,      /* BernoulliLoss :293-318   (labels 0/1, encoded 2y-1 in-kernel) */
  SE_LOSS_EXPONENTIAL = 7,    /* ExponentialLoss :265-291 (labels 0/1, encoded 2y-1 in-kernel) */
  SE_LOSS_LOGLOSS = 8         /* LogLoss(K) :196-263      (labels = class index, dim = K) */
};

/* ---- device slots (all fp32) ---------------------------------------------------------------- */
enum se_slot {
  SE_SLOT_Y = 0,      /* [n]        labels (Instance.label)                                   */
  SE_SLOT_W = 1,      /* [n]        instance weights (Instance.weight); absent => 1.0          */
  SE_SLOT_F = 2,      /* [dim][n]   running predictions  (GBMRegressor.scala:313, GBMClassifier.scala:294) */
  SE_SLOT_H = 3,      /* [dim][n]   directions = base model outputs this round (:405,:435)     */
  SE_SLOT_R = 4,      /* [dim][n]   pseudo-residuals = base-learner labels (:368-385)          */
  SE_SLOT_WOUT = 5,   /* [dim][n]   base-learner weights (newton: 1/2 h/S w, :379; the device holds 1/2 h w, se_download applies 1/S_dim) */
  SE_SLOT_VY = 6,     /* [nv]       validation labels                                          */
  SE_SLOT_VF = 7,     /* [dim][nv]  validation predictions (:324,:444-449)                     */
  SE_SLOT_VH = 8,     /* [dim][nv]  validation directions                                      */
  SE_SLOT_BW = 9,     /* [n]        boosting weights (BoostingClassifier.scala:168)            */
  SE_SLOT_PROBA = 10, /* [K][n]     base-model class probabilities (SAMME.R, :199-200)         */
  SE_SLOT_PRED = 11,  /* [n]        base-model predicted labels (SAMME, :232-233)              */
  SE_SLOT_P = 12,     /* [M][n] | [M][C][n]  stacked base-model outputs for Model.predict*     */
  SE_SLOT_RAW = 13,   /* [C][n]     aggregated rawPrediction / regression prediction ([1][n])  */
  SE_SLOT_PROB = 14,  /* [C][n]     probability column                                         */
  SE_SLOT_LABEL = 15, /* [n]        prediction column of classifiers (argmax raw)              */
  SE_SLOT_X = 16,     /* [d][n]     feature matrix, column-major (on-device base-model predict) */
  SE_SLOT_VX = 17,    /* [d][nv]    validation feature matrix                                   */
  SE_SLOT_BAG = 18,   /* [n]        bag multiplicities of RDD.sample (0/1 without, Poisson counts with replacement) */
  SE_NUM_SLOTS = 19
};

/* ---- library / context ---------------------------------------------------------------------- */
SE_API int se_abi_version(void);
SE_API const char* se_last_error(const se_ctx* ctx); /* ctx may be NULL: last error of the calling thread */
SE_API int se_device_count(int* out);
SE_API int se_ctx_create(int device, se_ctx** out);
SE_API int se_ctx_destroy(se_ctx* ctx);
SE_API int se_ctx_sync(se_ctx* ctx);
SE_API int se_ctx_device(const se_ctx* ctx, int* device);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
SE_API int se_ctx_launch_count(const se_ctx* ctx, int64_t* out);
/* device milliseconds of the most recent compute entry point (CUDA events on the context stream) */
SE_API int se_ctx_last_ms(se_ctx* ctx, double* out);
/* enable/disable per-call CUDA-event timing (default off: no extra events on the stream) */
SE_API int se_ctx_set_timing(se_ctx* ctx, int on);
/* stopwatch on the context stream (CUDA events): start enqueues an event; stop enqueues a second
 * one, waits for it and returns the device milliseconds in between */
SE_API int se_ctx_timer_start(se_ctx* ctx);
SE_API int se_ctx_timer_stop(se_ctx* ctx, double* ms);
/* per-kernel-family device time (CUDA events bracketing each launch while kernel timing is on):
 * families are enum se_kernel_family; total_ms / launches accumulate until reset */
enum se_kernel_family {
  SE_KF_SQ_STATS = 0, SE_KF_EVAL = 1, SE_KF_UPDATE = 2, SE_KF_RESID = 3, SE_KF_MEAN_LOSS = 4,
  SE_KF_BOOST_REAL = 5, SE_KF_BOOST_ERR = 6, SE_KF_BOOST_UPD = 7, SE_KF_AGG = 8, SE_KF_TREE = 9,
  SE_KF_LINEAR = 10, SE_KF_OTHER = 11, SE_KF_COUNT = 12
};
SE_API int se_ctx_kernel_timing(se_ctx* ctx, int on);
SE_API int se_ctx_kernel_time(se_ctx* ctx, int family, double* total_ms, int64_t* launches);
SE_API int se_ctx_kernel_time_reset(se_ctx* ctx);
/* Tunables and diagnostics by name (doubles).  Settable: "fused_round" (-1 auto by shard size / 0 / 1: squared-loss
 * round in ONE cooperative launch), "fused_round_max_rows", "fused_ctas_per_sm", "fused_prefetch_mb", "ls_mode" (non-squared Brent line
 * search: 0 = one launch per evaluation, 1 = one persistent launch with Brent on the device [default], 2 = host Brent
 * over single-evaluation launches of the persistent kernel — bit-identical to 1, for tests), "ls_resident",
 * "ls_ctas_per_sm", "ls_ring" (cp.async ring stages for the streamed tiles, 0 = register prefetch [default]), "l2_persist", "l2_persist_frac", "peer_timeout_ms" (spin bound of the fused peer exchange,
 * 0 = forever), "alternate_passes", "l2_hints", "ctas_per_sm", "host_mirror", "tree_bins" (uint8 rank matrix for tree
 * walks), "tree_mask" (all-nodes kernel for trees of <= 64 internal nodes), "wm_fast" (weighted median, M <= 64 and
 * weights >= 0: keys-only sort + margin-checked model-order sums, exact kernel for the deferred rows), "wm_list_cap"
 * (deferred-row list capacity, 0 = rows / 4).  Read-only: "last_tree_binned", "last_tree_mask", "last_wm_mode" (0 exact,
 * 1 fast with margin, 2 equal weights), "last_wm_deferred" (synchronises), "last_round_fused",
 * "last_ls_workers", "last_ls_passes", "last_ls_hit_ratio", "last_fused_grid", "l2_persist_max_bytes",
 * "l2_window_max_bytes".  Unknown keys fail with SE_ERR_ARG. */
SE_API int se_ctx_set_option(se_ctx* ctx, const char* key, double value);
SE_API int se_ctx_get_option(const se_ctx* ctx, const char* key, double* value);
/* pinned (page-locked) host memory for the buffers handed to se_upload/se_download (JNI: wrap in a
 * direct ByteBuffer); pageable memory works too but is staged by the driver */
SE_API int se_host_alloc(int64_t bytes, void** out);
SE_API int se_host_free(void* ptr);

/* ---- row-shard communicator: replaces Spark treeAggregate/treeReduce (SURVEY.md §2) ---------- */
#define SE_COMM_ID_BYTES 128
SE_API int se_comm_unique_id(void* out, int bytes);
SE_API int se_comm_init(se_ctx* ctx, int nranks, int rank, const void* id, int bytes);
/* 1 when the fused NVLink all-reduce is active: every rank's mailbox is mapped into every process with CUDA
 * IPC and the last CTA of each reducing kernel exchanges the per-GPU sums over peer memory itself (no separate
 * NCCL launch).  0: NCCL all-reduce after the kernel (fallback when IPC mapping fails or SE_P2P_ALLREDUCE=0). */
SE_API int se_comm_p2p_active(const se_ctx* ctx, int* active);
/* A peer that does not launch the matching reduction within "peer_timeout_ms" (default 120 s; se_ctx_set_option)
 * makes the waiting rank POISON that reduction in every peer's mailbox, so that all ranks fail the same reduction
 * with SE_ERR_NCCL instead of disagreeing on its result.  The error is sticky until every rank calls this. */
SE_API int se_comm_clear_error(se_ctx* ctx);
SE_API int se_comm_destroy(se_ctx* ctx);
SE_API int se_comm_info(const se_ctx* ctx, int* nranks, int* rank);
/* sum-allreduce `count` doubles held on the host across ranks (no-op without a communicator) */
SE_API int se_comm_allreduce_host(se_ctx* ctx, double* values, int count);

/* ---- slots ---------------------------------------------------------------------------------- */
SE_API int se_slot_alloc(se_ctx* ctx, int slot, int64_t count);               /* count fp32 elements */
/* [rows][cols] slot; rows > 1 get a padded row stride `ld` (multiple of 32 floats = 128 B) so every
 * row starts 128-bit aligned.  se_upload/se_download offsets are LOGICAL (row*cols + col). */
SE_API int se_slot_alloc2d(se_ctx* ctx, int slot, int64_t rows, int64_t cols);
SE_API int se_slot_layout(const se_ctx* ctx, int slot, int64_t* rows, int64_t* cols, int64_t* ld);
SE_API int se_slot_free(se_ctx* ctx, int slot);
SE_API int se_slot_info(const se_ctx* ctx, int slot, void** device_ptr, int64_t* count);
SE_API int se_upload(se_ctx* ctx, int slot, const float* host, int64_t count, int64_t offset);
SE_API int se_upload_f64(se_ctx* ctx, int slot, const double* host, int64_t count, int64_t offset);
/* Ingest of a feature partition (SURVEY §8f-4): `host` is ROW-major [n_rows][d] (the layout of Spark's dense
 * feature vectors); it lands in rows [row_offset, row_offset + n_rows) of the COLUMN-major [d][n] slot
 * (SE_SLOT_X / SE_SLOT_VX).  Chunked and double buffered: chunk c+1 is staged into pinned memory (or copied
 * straight from `host` when it is already page-locked) while chunk c is in flight over PCIe and chunk c-1 is
 * being transposed on the device by a 32x32 shared-memory tile kernel. */
SE_API int se_upload_rowmajor(se_ctx* ctx, int slot, const float* host, int64_t n_rows, int d, int64_t row_offset);
SE_API int se_download(se_ctx* ctx, int slot, float* host, int64_t count, int64_t offset);
/* download slot*scale (e.g. BoostingClassifier.scala:186 weight = boostingWeight / sumWeights) */
SE_API int se_download_scaled(se_ctx* ctx, int slot, double scale, float* host, int64_t count, int64_t offset);
SE_API int se_fill(se_ctx* ctx, int slot, float value, int64_t count, int64_t offset);
SE_API int se_copy_slot(se_ctx* ctx, int dst_slot, int src_slot);
/* deterministic counter-based synthetic fill (bench/tests): kind 0 uniform[a,b), 1 normal(a,b),
 * 2 integer uniform in [a,b) stored as float, 3 bernoulli(p=a) 0/1 */
SE_API int se_fill_synthetic(se_ctx* ctx, int slot, int kind, uint64_t seed, double a, double b,
                      int64_t count, int64_t offset);
/* Exact q-quantile (the ceil(q·N)-th smallest of the GLOBAL N values, i.e. what Spark's approxQuantile
 * returns as relativeError -> 0) by 4 radix-select passes over the fp32 keys; histograms are all-reduced.
 * which = 0: values of `slot`; which = 1: |Y − F| on the train shard (huber δ, regression/GBMRegressor.scala:
 * 342-353).  Used for DummyRegressor median/quantile inits (:119-125) and huber's δ (:305-308). SURVEY §8f-3 */
SE_API int se_quantile(se_ctx* ctx, int which, int slot, int64_t count, double q, double* out);
/* Σ slot[0..count) in fp64, all-reduced (BoostingClassifier.scala:175,269 sumWeights) */
SE_API int se_slot_sum(se_ctx* ctx, int slot, int64_t count, double* out);

/* ---- GBM inner loop: regression/GBMRegressor.scala:340-469, classification/GBMClassifier.scala:325-483 */
/* Declares the problem: local rows, validation rows, dim (1 or K), loss.  Allocates
 * Y,F,H,R (+W,WOUT when has_weights or newton is later used) and VY,VF,VH when n_valid > 0. */
SE_API int se_gbm_configure(se_ctx* ctx, int64_t n_train, int64_t n_valid, int dim, int loss,
                     double param, int has_weights);
SE_API int se_gbm_set_loss_param(se_ctx* ctx, double param); /* huber: delta re-estimated each round (:342-353) */
/* Row sub-sampling (regression/GBMRegressor.scala:357-359, classification/GBMClassifier.scala:329-331; SURVEY §8f-4):
 * on != 0 allocates SE_SLOT_BAG[n]; the host uploads the multiplicity of every train row in the bag (the
 * sample itself is Spark's RDD.sample — same seed every round, reference quirk 3).  While enabled, the
 * line-search sums (eval / stats: lossSum, weightSum, gradSum) and newton's Σ max(H,1e-2) run over the bag;
 * the F update, the fused residuals and the train loss stay on the full train set (reference quirk 4). */
SE_API int se_gbm_set_bag(se_ctx* ctx, int on);
/* pseudo-residuals from the current F (GBMRegressor.scala:368-385, GBMClassifier.scala:337-375).
 * newton=0: R=-g (base-learner weight stays the instance weight W).  newton=1 (loss has a hessian):
 * h=max(H,1e-2), S=Σh (all-reduced), R=-g/h, WOUT=1/2·h/S·w; sum_hess[dim] receives S. */
SE_API int se_gbm_pseudo_residuals(se_ctx* ctx, int newton, double* sum_hess);
/* GBMLossAggregator + RDDLossFunction.calculate (GBMLoss.scala:50-74): for coefficients alpha[dim]
 * returns loss = lossSum/weightSum (lossSum counted dim times per row: reference quirk) and
 * grad[dim] = gradSum/weightSum (grad may be NULL).  One streaming pass over Y,F,H. */
SE_API int se_gbm_linesearch_eval(se_ctx* ctx, const double* alpha, double* loss, double* grad);
/* squared loss only: the three sufficient statistics of the line-search parabola in one pass,
 * stats = {Σ(y-F)², Σh(y-F), Σh², weightSum}; objective(α) = (s0 - 2α s1 + α² s2) / (2 s3).
 * When SE_SLOT_R is current (after se_gbm_pseudo_residuals or a fused update) the pass reads r = y-F and h only
 * (8 B/row, bit-identical); any write to Y/F/R through this ABI reverts to reading y, F, h (12 B/row). */
SE_API int se_gbm_linesearch_stats(se_ctx* ctx, double* stats4);
/* F_j += step_j·H_j (GBMRegressor.scala:437-441; GBMClassifier.scala:437-448), fused with what the
 * next round needs: flags select extra outputs computed from the NEW F in the same pass. */
#define SE_UPD_RESIDUAL 1 /* R = -g(y,F')             (next round's pseudo-residuals, gradient mode) */
#define SE_UPD_NEWTON 2   /* R = -g/h, WOUT = 1/2·h/S·w, S returned in sum_hess (newton mode)          */
#define SE_UPD_LOSS 4     /* loss_sum = Σ loss(y,F')  (train loss of the new F, all-reduced)          */
SE_API int se_gbm_update(se_ctx* ctx, const double* step, int flags, double* loss_sum, double* sum_hess);
/* mean over rows of loss(y,F) on the train (which=0) or validation (which=1) shard
 * (GBMRegressor.scala:330-335,451-456) */
SE_API int se_gbm_mean_loss(se_ctx* ctx, int which, double* out);
/* VF_j += step_j·VH_j then mean validation loss (GBMRegressor.scala:444-456) */
SE_API int se_gbm_update_validation(se_ctx* ctx, const double* step, double* mean_loss);
/* Whole line search natively for dim == 1: commons-math3 Brent (GBMRegressor.scala:311,413-421) over
 * se_gbm_linesearch_eval; for squared loss Brent runs over the closed-form parabola built from
 * se_gbm_linesearch_stats (one pass, identical objective values up to rounding). */
SE_API int se_gbm_linesearch_brent(se_ctx* ctx, double lo, double hi, double start, double rel,
                            double abs_tol, int max_eval, double* alpha, double* loss, int* n_eval);
/* One boosting round for dim == 1 in a single call (GBMRegressor.scala:398-442): Brent line search
 * (optimized != 0; else alpha = 1), weight = learning_rate·alpha, then se_gbm_update(weight, flags).
 * Same results as se_gbm_linesearch_brent + se_gbm_update; saves the host round-trips between them. */
SE_API int se_gbm_round(se_ctx* ctx, double learning_rate, int optimized, double tol, int max_iter, int flags,
                        double* alpha, double* loss_sum, int* n_eval);
/* Opt-in fast line search for dim == 1 losses with a hessian (squared, bernoulli, exponential, logcosh): each
 * pass also returns the curvature Σ h²·H, and a safeguarded Newton iteration on [lo,hi] converges in ~4-6
 * passes instead of Brent's 20-40.  NOT the reference's optimiser: it returns a minimiser within the same
 * tolerance (|Δα| <= rel·|α| + abs) but with different iterates; Brent stays the default (drop-in parity). */
SE_API int se_gbm_linesearch_eval2(se_ctx* ctx, double alpha, double* loss, double* d1, double* d2);
SE_API int se_gbm_linesearch_newton(se_ctx* ctx, double lo, double hi, double start, double rel, double abs_tol,
                                    int max_eval, double* alpha, double* loss, int* n_eval);
/* squared loss, no host round-trip: stats pass -> (allreduce) -> closed-form α*=clip(s1/s2,0,100)
 * on device -> F += lr·α*·H fused with R=-g and Σloss.  Results are fetched with
 * se_gbm_round_result(); rounds may be enqueued back-to-back (or captured in a CUDA graph). */
SE_API int se_gbm_round_squared_async(se_ctx* ctx, double learning_rate);
SE_API int se_gbm_round_result(se_ctx* ctx, double* alpha, double* loss_sum);

/* univariate Brent (commons-math3 3.6.1 BrentOptimizer semantics) exposed for host optimisers */
typedef double (*se_fn1)(double x, void* user);
SE_API int se_brent_minimize(se_fn1 f, void* user, double lo, double hi, double start, double rel,
                      double abs_tol, int max_eval, double* x_out, double* f_out, int* n_eval);

/* ---- BoostingClassifier weight update: classification/BoostingClassifier.scala:168-269 ------- */
/* allocates Y, BW and PROBA[K][n] (real) or PRED[n] (discrete) */
SE_API int se_boost_configure(se_ctx* ctx, int64_t n, int num_classes, int real);
/* SAMME.R (:198-230) in one pass: est_err = Σ wₙ·1[argmax p ≠ y], BW ← wₙ·exp(-(K-1)/K·Σ c_k log max(p_k,ε)),
 * new_sum = Σ BW.  wₙ = BW/sum_w. */
SE_API int se_boost_real_update(se_ctx* ctx, double sum_w, double* est_err, double* new_sum);
/* SAMME (:231-260): error pass, then update pass BW ← wₙ·(1/β)^err */
SE_API int se_boost_discrete_error(se_ctx* ctx, double sum_w, double* est_err);
SE_API int se_boost_discrete_update(se_ctx* ctx, double sum_w, double beta, double* new_sum);

/* ---- BoostingRegressor (AdaBoost.R2) weight update: regression/BoostingRegressor.scala:205-263 (§8f-2) */
enum se_r2_loss { SE_R2_EXPONENTIAL = 0, SE_R2_LINEAR = 1, SE_R2_SQUARED = 2 }; /* :97-106 */
/* allocates Y, BW and PRED[n] */
SE_API int se_boostreg_configure(se_ctx* ctx, int64_t n);
/* maxError = max_i |y_i − pred_i| (:231-234), max-all-reduced across shards */
SE_API int se_boostreg_max_error(se_ctx* ctx, double* max_error);
/* estimatorError = Σ wₙ·loss(|y−pred| / maxError) (loss(|y−pred|) when maxError == 0), wₙ = BW/sum_w (:236-249) */
SE_API int se_boostreg_error(se_ctx* ctx, double sum_w, int loss_type, double max_error, double* est_err);
/* BW ← wₙ·β^(1−loss) (:256-260); new_sum = Σ BW (:263) */
SE_API int se_boostreg_update(se_ctx* ctx, double sum_w, int loss_type, double max_error, double beta,
                              double* new_sum);

/* ---- ensemble Model.predict / predictRaw aggregation (SURVEY.md §3.4) ------------------------ */
enum se_agg_kind {
  SE_AGG_GBM_REGRESSOR = 0,      /* regression/GBMRegressor.scala:531-539   init + Σ a_m P[m]     */
  SE_AGG_BAGGING_REGRESSOR = 1,  /* regression/BaggingRegressor.scala:221-228   (Σ P[m]) / M      */
  SE_AGG_GBM_CLASSIFIER = 2,     /* classification/GBMClassifier.scala:564-589  (+ loss-specific prob) */
  SE_AGG_BAGGING_SOFT = 3,       /* classification/BaggingClassifier.scala:260-287 soft vote      */
  SE_AGG_BAGGING_HARD = 4,       /* ... hard vote: P holds predicted labels [M][n]                */
  SE_AGG_BOOSTING_REAL = 5,      /* classification/BoostingClassifier.scala:348-364               */
  SE_AGG_BOOSTING_DISCRETE = 6,  /* classification/BoostingClassifier.scala:366-382               */
  SE_AGG_BOOSTING_REG_MEDIAN = 7, /* regression/BoostingRegressor.scala:333-337 + ensemble/Utils.scala:26-40 (weighted median) */
  SE_AGG_BOOSTING_REG_MEAN = 8    /* regression/BoostingRegressor.scala:339-342  dot(p, w) / Σw    */
};
/* allocates P ([M][n] or [M][width][n]), RAW, PROB and LABEL for classifiers.
 * width: GBM classifier = dim; soft/real = num_classes; others 1. */
SE_API int se_agg_configure(se_ctx* ctx, int kind, int num_models, int num_classes, int dim, int loss,
                     int64_t n);
/* runs the aggregation over P.  weights: [M] (GBM regressor, boosting discrete) or [M][dim]
 * (GBM classifier) or NULL; init: [dim] or NULL. Fills RAW (+PROB, LABEL for classifiers). */
SE_API int se_agg_run(se_ctx* ctx, const double* weights, const double* init);

/* ---- row sub-sampling: Spark's sampler restated for the host side that has no Spark ------------- */
/* Multiplicities (0/1) of RDD.sample(withReplacement = false, fraction, seed) for `n` rows that sit in Spark partition
 * `partition` (regression/GBMRegressor.scala:357-359): java.util.Random(seed) -> per-partition seed ->
 * XORShiftRandom -> BernoulliSampler (gap sampling for fraction <= 0.4).  Host-only, no GPU involved; restated from the
 * Spark 3.3.1 sources and UNPINNED (no Spark here) — a Spark host uploads the multiplicities Spark drew instead. */
SE_API int se_spark_bernoulli_sample(int64_t seed, double fraction, int64_t n, int partition, float* counts);

/* ---- on-device base-model evaluation over column-major X (SURVEY.md §8f-1) ------------------- */
/* Decision tree in array form (node i: feature[i] < 0 => leaf with value[i]; else go left when
 * x[feature[i]] <= threshold[i], as Spark's ContinuousSplit.shouldGoLeft).  Writes out_slot row
 * `out_row` ([.][n]) from X (which = 0: SE_SLOT_X, 1: SE_SLOT_VX). `subspace` maps model feature index
 * -> column of X (HasSubBag.slice, ensemble/HasSubBag.scala:81-84) or NULL for identity.
 * The arrays must describe a TREE rooted at node 0: a node reached twice (cycle / shared child) fails with
 * SE_ERR_ARG before anything is launched.  Thresholds: the device compares the fp32 feature with the fp32 threshold;
 * pass the LARGEST float <= the fp64 threshold (round toward -inf: learners.py / FlatTree do) — then `x <= thr`
 * decides exactly like the JVM for every feature value that is itself a float (which is what HBM holds).  A fp64
 * feature value strictly between that float and the fp64 threshold can still change sides: the resident feature
 * matrix is fp32 by contract (north_star), so transform with the model on the same fp32 features. */
SE_API int se_tree_predict(se_ctx* ctx, int which, int n_nodes, const int32_t* feature,
                    const float* threshold, const int32_t* left, const int32_t* right,
                    const float* value, const int32_t* subspace, int n_subspace, int out_slot,
                    int out_row);
/* Classification tree: every node carries a vector of n_out values (`values` is [n_nodes][n_out], e.g. the leaf's
 * class probabilities = predictProbability); rows 0..n_out-1 of out_slot ([n_out][n]) are written.  Feeds
 * SE_SLOT_PROBA for SAMME.R (BoostingClassifier.scala:199-200) without moving K x n probabilities over PCIe. */
SE_API int se_tree_predict_multi(se_ctx* ctx, int which, int n_nodes, const int32_t* feature,
                                 const float* threshold, const int32_t* left, const int32_t* right,
                                 const float* values, int n_out, const int32_t* subspace, int n_subspace,
                                 int out_slot);
/* A whole ensemble of regression trees in ONE pass: out[row] = init + Σ_t weights[t] · tree_t(x_row), accumulated in
 * fp64 in model order — GBMRegressionModel.predict (regression/GBMRegressor.scala:531-539); with weights 1/M and
 * init 0, BaggingRegressionModel.predict (regression/BaggingRegressor.scala:221-228).  The trees are concatenated: tree t
 * owns nodes [offsets[t], offsets[t+1]) of the five node arrays, child indices are TREE-LOCAL, `feature` holds GLOBAL
 * columns of X (map each member's subspace, ensemble/HasSubBag.scala:81-84, before the call), weights NULL = all 1.
 * Runs over the uint8 rank matrix (see se_tree_predict; fails with SE_ERR_STATE when a column needs more than 255
 * thresholds: evaluate the members with se_tree_predict + se_agg_run then): the ranks of every column the forest uses
 * are staged once per 256-row tile in shared memory and every tree is walked out of shared memory — no [M][n]
 * intermediate.  Forests larger than the shared-memory budget run in chunks of trees (out accumulates in fp32
 * between chunks).  Same tree / threshold contract as se_tree_predict. */
SE_API int se_forest_predict(se_ctx* ctx, int which, int n_trees, const int32_t* offsets, const int32_t* feature,
                             const float* threshold, const int32_t* left, const int32_t* right, const float* value,
                             const double* weights, double init, int out_slot, int out_row);
/* A classifier ensemble of trees in ONE pass over the uint8 rank matrix of X (which = 0) or VX (which = 1), with no
 * [M][K][n] member outputs.  Writes SE_SLOT_RAW [C][n], SE_SLOT_PROB [C][n] and SE_SLOT_LABEL [n] exactly as
 * se_agg_configure(kind, M, num_classes, dim, loss, n) + se_agg_run(weights, init) would from the members' outputs.
 * It allocates those three slots itself (n = columns of the feature slot) and never allocates SE_SLOT_P.
 * Trees are concatenated as in se_forest_predict (offsets, tree-local children, GLOBAL columns).  Per kind:
 *   SE_AGG_GBM_CLASSIFIER    M·dim trees, tree t = models(t / dim)(t % dim); leaf = regression value (leaf_width 1);
 *                            weights [M][dim] (required), init [dim] or NULL (zeros)
 *   SE_AGG_BAGGING_SOFT      M trees; leaf = class probabilities (leaf_width K); weights, init ignored
 *   SE_AGG_BOOSTING_REAL     M trees; leaf = class probabilities (leaf_width K), summed as log(max(p, 2^-52)) formed
 *                            once per leaf in fp64; weights, init ignored
 *   SE_AGG_BAGGING_HARD      M trees; leaf = predicted label (leaf_width 1, K <= 65536); weights, init ignored
 *   SE_AGG_BOOSTING_DISCRETE M trees; leaf = predicted label (leaf_width 1, K <= 65536); weights [M] (required)
 * `leaf` is [total nodes][leaf_width] (internal nodes' entries are ignored).  A label leaf that is not an integer in
 * [0, K), another kind, a leaf_width that does not match the kind, a node array that is not a tree or a column outside X
 * fail with SE_ERR_ARG; a column that needs more than 255 thresholds (or no feature slot) with SE_ERR_STATE — evaluate
 * the members with se_tree_predict* + se_agg_run then.  The class sums accumulate in fp64 in model order inside a chunk
 * of trees and in RAW (fp32) between chunks; option last_forest_chunks reports the chunk count. */
SE_API int se_forest_classify(se_ctx* ctx, int which, int kind, int num_classes, int dim, int loss,
                              int n_trees, const int32_t* offsets, const int32_t* feature, const float* threshold,
                              const int32_t* left, const int32_t* right, const float* leaf, int leaf_width,
                              const double* weights, const double* init);
/* AdaBoost.R2's weighted median of tree members in ONE pass over the uint8 rank matrix of X (which = 0) or VX (which = 1):
 * row out_row of out_slot receives Utils.weightedMedian([tree_t(x)]_t, weights) for every row, with no [M][n] member
 * outputs.  Trees are concatenated as in se_forest_predict (offsets, tree-local children, GLOBAL columns, `value` = the
 * leaf value per node), in model order; equal member values are ordered by model index (the reference's stable sortBy).
 * The output is bit-identical to se_tree_predict of every member into row t of SE_SLOT_P followed by
 * se_agg_configure(SE_AGG_BOOSTING_REG_MEDIAN, M, ...) + se_agg_run(weights), for every weight vector (zero, negative,
 * equal, half-weight ties) and with option wm_fast on or off: it is a selection among the fp32 leaf values.  The weights
 * choose the mode exactly as in se_agg_run (last_wm_mode: 0 exact, 1 fast + margin, 2 equal weights); in mode 1 the rows
 * inside the rounding margin take the exact pick in the same thread and last_wm_deferred counts them.
 * Sets last_forest_chunks = 1 and last_tree_binned = 1.
 * SE_ERR_ARG: a null pointer (weights included), a node array that is not a tree, a column outside X.
 * SE_ERR_STATE: no feature slot, an output slot whose column count differs from the feature slot's, a column that needs
 * more than 255 thresholds, more than 64 trees, or a forest that does not fit ONE chunk of the forest kernel's shared
 * memory (nodes, leaf values, ranks and parked leaves within 216 KB) — evaluate the members with se_tree_predict +
 * se_agg_run then. */
SE_API int se_forest_weighted_median(se_ctx* ctx, int which, int n_trees, const int32_t* offsets, const int32_t* feature,
                                     const float* threshold, const int32_t* left, const int32_t* right, const float* value,
                                     const double* weights, int out_slot, int out_row);
/* linear model: out = intercept + Σ_j coef[j]·X[subspace[j]] */
SE_API int se_linear_predict(se_ctx* ctx, int which, int n_coef, const float* coef, float intercept,
                      const int32_t* subspace, int out_slot, int out_row);

#ifdef __cplusplus
}
#endif
#endif /* SE_ABI_H */
