// se_kernels.h — host-callable launchers of the sm_100a kernels (internal to libse_b200.so).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "se_common.cuh"

namespace se {

constexpr int kMaxDim = 64;  // LogLoss classes served by the specialised kernels: per-class sums reduced in one kernel (kMaxRed, mailbox width)
constexpr int kMaxDimGeneric = 16384;  // beyond kMaxDim: the general kernels of se_gbm_generic.cu (shared-memory accumulators)

// ---- GBM (se_gbm.cu) -------------------------------------------------------------------------
enum GbmMode {
  GBM_RESID = 0,         // R = -g(y,F)
  GBM_RESID_NEWTON = 1,  // R = -g/hc, WOUT = 1/2 hc w (unnormalised), Σhc
  GBM_EVAL = 2,          // p = F + a h : Σloss, Σ h g      (GBMLossAggregator.add)
  GBM_UPDATE = 3,        // F += s h : Σloss(F')
  GBM_UPDATE_RESID = 4,  // + R = -g(y,F')
  GBM_UPDATE_NEWTON = 5, // + R = -g/hc, WOUT = 1/2 hc w, Σhc
  GBM_MEAN_LOSS = 6,     // Σloss(y,F)
  GBM_SQ_STATS = 7,      // squared: Σ(y-F)², Σh(y-F), Σh²
  GBM_EVAL_LOSS = 8      // p = F + a h : Σloss only (Brent needs the objective value, not its gradient)
};

struct GbmArgs {
  const float* y = nullptr;
  const float* w = nullptr;  // nullable: unit weights
  const float* bag = nullptr;  // nullable: per-row bag multiplicities (RDD.sample counts) for line search / newton S
  float* F = nullptr;
  const float* h = nullptr;
  float* r = nullptr;
  float* wout = nullptr;
  int64_t n = 0;
  int64_t ld = 0;  // row stride of the [dim][n] arrays
  int dim = 1;
  float param = 0.f;
  float coef[kMaxDim] = {0};  // alpha (eval) or step (update), per dim
  // squared-loss device-resident step: step = lr * clip(stats[1]/stats[2], 0, 100) when non-null
  const double* dev_stats = nullptr;
  float lr = 1.f;
  // step = (float)(lr64 * *dev_alpha) when non-null: alpha comes from the on-device line search (se_brent.cu)
  const double* dev_alpha = nullptr;
  double lr64 = 1.0;
  int stages = 1;  // tiled logloss kernel: shared-memory stages (1, or 2 for experiments)
  int stats_from_r = 0;  // squared-loss statistics read the current residual slot r = y - F (8 B/row) instead of y, F (12 B/row)
  int l2_hints = 0; // L2-sized shard: evict_first for the arrays the next pass does not re-read (se_common.cuh)
  int reverse = 0; // walk the tiles from the end: consecutive passes alternate direction so the tail of one
                   // pass (still in the 126 MB L2) is the head of the next
  RedWs ws{};
};

// reduction outputs (ws.out): scalar losses: [0]=Σloss [1]=Σ h·g or Σhc ; SQ_STATS: [0..2]
// logloss: [0]=Σloss, [1..K]=Σ h_j g_j  or Σhc_j
cudaError_t launch_gbm(int loss, int mode, const GbmArgs& a, int ctas_per_sm, int sms,
                       cudaStream_t stream);
// line-search view for the binary scalar losses: u = (2y-1)·F, v = (2y-1)·h (exact sign flips), so that every
// Brent evaluation reads two arrays instead of three (launch_gbm GBM_EVAL with y == nullptr, F = u, h = v)
cudaError_t launch_gbm_pack_signed(const float* y, const float* F, const float* h, float* u, float* v, int64_t n,
                                   int sms, cudaStream_t stream);
// LogLoss(K) for K > kMaxDim (se_gbm_generic.cu): coefficients, per-CTA partials [grid][K+1] and the K+1 sums live in
// device buffers sized for K; the cross-GPU sum of `out` is an NCCL all-reduce issued by the caller
struct GenericArgs {
  const float* coef = nullptr;  // device [K]
  double* partials = nullptr;   // device [grid][K+1]
  double* out = nullptr;        // device [K+1]
};
cudaError_t launch_gbm_logloss_generic(int mode, const GbmArgs& a, const GenericArgs& ga, int grid, cudaStream_t stream);
// LogLoss(K), wide K: 2-D TMA tiles of 256 rows x K classes, four rows per thread (se_gbm_tiled.cu)
cudaError_t launch_gbm_logloss_tiled(int mode, const GbmArgs& a, int sms, cudaStream_t stream);
// squared-loss line search on the device: Brent over the parabola of stats[0..2]; out[0] = alpha, out[1] = objective,
// out[2] = evaluations (negative: MaxEval exceeded); out_host (mapped pinned memory) is optional
cudaError_t launch_brent_parabola(const double* stats, double wsum, double lo, double hi, double start, double rel,
                                  double abs_tol, int max_eval, double* out_dev, double* out_host, cudaStream_t stream);
// squared-loss round result: out[0] = alpha*, computed on device from stats (for se_gbm_round_result)
cudaError_t launch_sq_alpha(const double* stats, double* out_alpha, cudaStream_t stream);

// ---- whole-round / whole-line-search cooperative kernels (se_gbm_fused.cu) ----------------------
// Device-side rendezvous of the cooperative kernels (owned by the context, zero-initialised).
struct FusedSync {
  unsigned long long flag;  // epoch published by the coordinating CTA / warp (monotonic across launches)
  double x;                 // published with the flag: the step (round kernel) or the next abscissa (line search)
  int cmd;                  // line search: 0 = evaluate x, 1 = stop
  int pad;
  unsigned int arrive;      // line search: worker arrival counter (reset by the coordinator)
  unsigned int counter_b;   // round kernel: ticket of the second (loss) reduction
};

// One squared-loss boosting round in one launch: statistics -> (cross-GPU sum) -> Brent -> update + residual + loss.
struct SqRoundArgs {
  const float* y = nullptr;
  float* F = nullptr;
  const float* h = nullptr;
  float* r = nullptr;
  const float* bag = nullptr;  // nullable: bag multiplicities for the line-search statistics
  int64_t n = 0;
  int stats_from_r = 0;
  int l2_hints = 0;
  int l2_mode = 0;         // 0: evict_normal / evict_first hints; 1: evict_last on r and h (experiment)
  int timing = 0;          // write %globaltimer stamps (us) to out[10..13]: start, statistics folded, step published, end
  int prefetch_tiles = 0;  // y/F tiles of the update phase each CTA prefetches into L2 while it waits for the step
  double lr = 1.0, wsum = 1.0;                                   // learning rate, Σw (objective scale)
  double lo = 0.0, hi = 100.0, start = 1.0, rel = 1e-6, abs_tol = 1e-6;
  int max_eval = 100;
  RedWs ws_a{};  // statistics: out = `out`, no host mirror
  RedWs ws_b{};  // loss (only when it is reduced over the rows: bags): out = out + 8, host mirror + ticket
  double* out = nullptr;       // [0..2] statistics, [4] alpha, [5] objective, [6] +-evaluations, [8] Σloss
  double* host_res = nullptr;  // mapped host copy of out[0..6] (nullable)
  // loss-from-statistics mode: the Brent thread also serves the host (final value + ticket) before the update phase ends
  double* host_final = nullptr;
  volatile unsigned long long* host_flag = nullptr;
  unsigned long long host_ticket = 0;
  FusedSync* sync = nullptr;
  unsigned long long epoch = 0;
};
cudaError_t launch_gbm_round_sq_fused(const SqRoundArgs& a, int write_r, int loss_reduce, int sms, int max_ctas_per_sm,
                                      cudaStream_t stream, int* grid_out, void* window_base = nullptr, size_t window_bytes = 0);

// Brent's whole line search for a dim-1 scalar loss in one launch (persistent workers + coordinator warp).
struct LsArgs {
  const float* y = nullptr;
  const float* F = nullptr;
  const float* h = nullptr;
  float* u = nullptr;  // binary losses: signed view written by the first evaluation, read by the others
  float* v = nullptr;
  int64_t n = 0;
  float param = 0.f;
  double wsum = 1.0;
  double lo = 0.0, hi = 100.0, start = 1.0, rel = 1e-6, abs_tol = 1e-6;
  int max_eval = 100;
  int timing = 0;        // diagnostics: out[4] = us spent in worker passes, out[5] = us in fold + cross-GPU exchange
  int single = 0;        // evaluate the objective at `start` once (host-driven search over the same kernel)
  int first_parity = 0;  // tile direction of evaluation e is (first_parity + e) & 1
  int resident_tiles = 0;
  int ring_stages = 0;   // > 0: streamed tiles go through a per-thread cp.async ring of this many stages in shared memory
  double* partials = nullptr;
  FusedSync* sync = nullptr;
  unsigned long long epoch0 = 0;
  RedWs ws{};            // peer exchange (seq = sequence of the FIRST evaluation) and host mirror
  double* out = nullptr; // [0] alpha, [1] objective, [2] +-evaluations (negative: MaxEval exceeded), [3] passes run
};
struct LsLaunch {
  int max_ctas_per_sm = 4;
  int resident = 1;             // keep each worker's first tiles in shared memory
  int ring = 0;                 // cp.async ring stages for the streamed tiles: 0 off (register prefetch), 2..4
  void* window_base = nullptr;  // L2 access-policy window (persisting) over the packed view
  size_t window_bytes = 0;
  float hit_ratio = 0.f;
};
bool gbm_linesearch_persist_supported(int loss);
bool gbm_linesearch_persist_packed(int loss);
cudaError_t launch_gbm_linesearch_persist(int loss, const LsArgs& a, int sms, const LsLaunch& cfg, cudaStream_t stream,
                                          int* workers_out);

// ---- Boosting (se_boost.cu) ------------------------------------------------------------------
struct BoostArgs {
  const float* y = nullptr;
  float* w = nullptr;         // updated in place
  const float* proba = nullptr;  // [K][n]
  const float* pred = nullptr;   // [n]
  int64_t n = 0, ld = 0;
  int K = 2;
  float inv_sum_w = 1.f;
  float inv_beta = 1.f;
  RedWs ws{};
};
cudaError_t launch_boost_real(const BoostArgs& a, int ctas_per_sm, int sms, cudaStream_t s);   // out: [0]=err [1]=Σw'
cudaError_t launch_boost_discrete_error(const BoostArgs& a, int ctas_per_sm, int sms, cudaStream_t s);  // out[0]
cudaError_t launch_boost_discrete_update(const BoostArgs& a, int ctas_per_sm, int sms, cudaStream_t s); // out[0]=Σw'
cudaError_t launch_sum(const float* x, int64_t n, const RedWs& ws, int ctas_per_sm, int sms,
                       cudaStream_t s);  // out[0]
// out[0] = Σ a_i·b_i (b nullable: Σ a_i)
cudaError_t launch_dot(const float* a, const float* b, int64_t n, const RedWs& ws, int ctas_per_sm, int sms,
                       cudaStream_t s);
// AdaBoost.R2 (regression/BoostingRegressor.scala:225-263). loss_type 0 exponential, 1 linear, 2 squared.
struct BoostRegArgs {
  const float* y = nullptr;
  const float* pred = nullptr;
  float* w = nullptr;  // updated in place by the update kernel
  int64_t n = 0;
  int loss_type = 0;
  float inv_sum_w = 1.f;
  float inv_max_err = 1.f;  // 1/maxError, or 1 when maxError == 0 (:236-242)
  float log2_beta = 0.f;
  RedWs ws{};
};
cudaError_t launch_boostreg_max(const BoostRegArgs& a, int ctas_per_sm, int sms, cudaStream_t s);     // out[0] = max|y-pred|
cudaError_t launch_boostreg_error(const BoostRegArgs& a, int ctas_per_sm, int sms, cudaStream_t s);   // out[0] = Σ wₙ·loss
cudaError_t launch_boostreg_update(const BoostRegArgs& a, int ctas_per_sm, int sms, cudaStream_t s);  // out[0] = Σ w'

// ---- Aggregation (se_agg.cu) -----------------------------------------------------------------
struct AggArgs {
  int kind = 0;
  const float* P = nullptr;  // [M][width][n] with row stride ld
  float* raw = nullptr;      // [C][n]
  float* prob = nullptr;     // [C][n] (classifiers)
  float* label = nullptr;    // [n]    (classifiers)
  const float* weights = nullptr;  // device [M] or [M][dim]
  const float* init = nullptr;     // device [dim]
  int M = 0, K = 0, dim = 1, loss = 0;
  int64_t n = 0, ld = 0, ld_out = 0;
  double sum_weights = 0.0;  // Σ a_m of the fp32-narrowed weights (boosting discrete epilogue, boosting-regressor mean)
  const double* weights64 = nullptr;  // device [M] fp64 (weighted median cumulative sums)
  int* bad_label = nullptr;           // raised (mapped host memory) when a vote is not a class index in [0, K)
  // weighted median fast path (M <= 64): 0 exact kernel only; 1 keys-only sort + model-order sums, rows within the
  // rounding margin of the half-weight deferred to the exact kernel through wm_list; 2 all weights equal (no margin)
  int wm_mode = 0;
  const double* weights64_host = nullptr;  // [M], the same values as weights64
  int32_t* wm_list = nullptr;              // [wm_cap] deferred rows
  unsigned int* wm_count = nullptr;        // number of deferred rows (may exceed wm_cap: the exact pass then covers all rows)
  unsigned int wm_cap = 0;
};
cudaError_t launch_agg(const AggArgs& a, int ctas_per_sm, int sms, cudaStream_t s);

// ---- base-model evaluators over column-major X (se_models.cu) --------------------------------
struct TreeArgs {
  const float* X = nullptr;  // [d][n], stride ld
  int64_t n = 0, ld = 0;
  int n_nodes = 0;
  const int32_t* feature = nullptr;  // device arrays [n_nodes]; feature already mapped through subspace
  const float* threshold = nullptr;
  const int32_t* left = nullptr;
  const int32_t* right = nullptr;
  const float* value = nullptr;      // [n_nodes][n_out]
  float* out = nullptr;              // n_out rows of stride ld_out
  int n_out = 1;                     // 1: regression value / label; K: class-probability vector of the leaf
  int64_t ld_out = 0;
};
cudaError_t launch_tree_predict(const TreeArgs& a, int sms, cudaStream_t s);
// uint8 rank matrix of X for the tree walk (se_models.cu): X8[col][i] = #{thresholds of col strictly below X[col][i]}
struct BinArgs {
  const float* X = nullptr;      // [d][ld]
  uint8_t* X8 = nullptr;         // [d][ld8]
  int64_t n = 0, ld = 0, ld8 = 0;
  const int32_t* cols = nullptr;     // device: the columns to (re)build, one per blockIdx.y
  const float* edges = nullptr;      // device [d][256]: sorted thresholds per column
  const int32_t* n_edges = nullptr;  // device [d]
};
cudaError_t launch_bin_columns(const BinArgs& a, int n_cols, int sms, cudaStream_t s);
// nodes: packed {x,y: byte offset of the column in X8 (64 bit); z: bin threshold | leaf << 31; w: left | right << 16}
// n_internal: number of internal nodes; mask_mode != 0 allows the all-nodes kernel for trees of <= 64 internal nodes
cudaError_t launch_tree_predict_binned(const TreeArgs& a, const uint8_t* X8, const uint4* nodes, int n_internal, int mask_mode,
                                       int sms, cudaStream_t s);
// A whole forest in ONE pass over the uint8 rank matrix: out = (accumulate ? out : init) + Σ_t w_t · tree_t(row)
// (GBMRegressionModel.predict, regression/GBMRegressor.scala:531-539; BaggingRegressionModel.predict,
// regression/BaggingRegressor.scala:221-228).  `blob` is the packed chunk of trees, copied verbatim into shared memory:
//   [0)            double   w[T]
//   [off_coloff)   uint64   byte offset of local column c in X8 (column * ld8), c < C
//   [off_nodes)    uint2    nodes: x = local column | rank threshold << 16 | leaf << 31, y = left | right << 16 (tree-local)
//   [off_treeoff)  int32    first node of tree t (T + 1 entries)
//   [off_values)   float    leaf value per node
//   [off_ranks)    uint8    (shared memory only) the tile's ranks, [C][256]
struct ForestArgs {
  const uint8_t* X8 = nullptr;
  int64_t n = 0, ld8 = 0;
  const unsigned char* blob = nullptr;
  int blob_bytes = 0;  // multiple of 16
  int T = 0, C = 0;
  int off_coloff = 0, off_nodes = 0, off_treeoff = 0, off_values = 0, off_ranks = 0;
  double init = 0.0;
  int accumulate = 0;
  float* out = nullptr;
};
constexpr int kForestTile = 256;              // rows per CTA tile (one row per thread)
constexpr int kForestSmemBudget = 54 * 1024;  // per CTA: four CTAs per SM (the walk is latency-bound: warps matter more than chunk size)
cudaError_t launch_forest_predict(const ForestArgs& a, int sms, cudaStream_t s);
// A classifier ensemble in ONE pass over the uint8 rank matrix: the stage-1 class sums of the aggregation (what
// agg_finalize reads from RAW) for classes [c0, c1), RAW[c][row] = start_c + Σ_t w_t · leaf contribution, fp64 in model
// order; start_c = RAW[c][row] for c in [acc0, acc1) (a sum an earlier chunk began), else init_c (GBM) or 0.
// Leaf kinds (mode): one value per leaf for the tree's own class (GBM: trees of class c are [cstart[c-c0], cstart[c-c0+1]));
// K values per leaf (class probabilities, or their logs for SAMME.R); a label per leaf (a vote of weight w_t).
// `blob` (copied verbatim into shared memory):
//   [0)            double   w[T]
//   [off_init)     double   init of classes c0.. (GBM only)
//   [off_coloff)   uint64   byte offset of local column c in X8 (column * ld8), c < C
//   [off_nodes)    uint2    nodes as in ForestArgs, a leaf's y = its ordinal among the tree's leaves
//   [off_treeoff)  int32    first node of tree t (T + 1 entries)
//   [off_lbase)    int32    first value of tree t's leaves in `leaves`
//   [off_cstart)   int32    GBM: first tree of class c0 + j (c1 - c0 + 1 entries)
//   [off_ranks)    uint8    (shared memory only) the tile's ranks, [C][256]
//   [off_parked)   uint16   (shared memory only) leaf ordinal (label for label leaves) per tree and row, [T][256]
enum { kForestScalarLeaves = 0, kForestVectorLeaves = 1, kForestLabelLeaves = 2 };
struct ForestClassArgs {
  const uint8_t* X8 = nullptr;
  int64_t n = 0, ld8 = 0;
  const unsigned char* blob = nullptr;
  int blob_bytes = 0;  // multiple of 16
  int T = 0, C = 0;
  int off_init = 0, off_coloff = 0, off_nodes = 0, off_treeoff = 0, off_lbase = 0, off_cstart = 0, off_ranks = 0, off_parked = 0;
  int mode = 0, K = 0;
  int c0 = 0, c1 = 0, acc0 = 0, acc1 = 0;
  const float* leaves = nullptr;  // device leaf table
  float* raw = nullptr;           // [C][ld_raw]
  int64_t ld_raw = 0;
};
cudaError_t launch_forest_classify(const ForestClassArgs& a, int sms, cudaStream_t s);
// The weighted median of a forest's members in ONE pass over the uint8 rank matrix (BoostingRegressionModel.predict
// with votingStrategy "median", regression/BoostingRegressor.scala:333-337): out[row] = the value se_agg_run
// (SE_AGG_BOOSTING_REG_MEDIAN) selects from the members' outputs, for T <= 64 trees that fit ONE chunk.  `blob` is
// ForestArgs' layout (w[T] are the fp64 weights, leaf value per node at off_values) followed in shared memory by
//   [off_ranks)    uint8    the tile's ranks, [C][256]
//   [off_parked)   uint32   the leaf value's order-preserving key (wm_key) per tree and row, [T][256]
// wm_mode 0: exact pick for every row; 1: keys-only sort + model-order bisection, rows inside the margin tau take the
// exact pick in the same thread and are counted in *deferred; 2: equal weights, fast path for every row.
struct ForestWmArgs {
  const uint8_t* X8 = nullptr;
  int64_t n = 0, ld8 = 0;
  const unsigned char* blob = nullptr;
  int blob_bytes = 0;  // multiple of 16
  int T = 0, C = 0;
  int off_coloff = 0, off_nodes = 0, off_treeoff = 0, off_values = 0, off_ranks = 0, off_parked = 0;
  int wm_mode = 0;
  const double* weights_host = nullptr;  // [T], host memory: the fast path's constant-bank operands
  unsigned int* deferred = nullptr;      // mode 1: rows that took the exact pick (zeroed by the launcher)
  float* out = nullptr;
};
cudaError_t launch_forest_wmedian(const ForestWmArgs& a, int sms, cudaStream_t s);
// The classifier aggregations' epilogue (se_agg.cu agg_finalize_kernel) over the stage-1 sums already in raw[C][ld]:
// raw, prob and label as se_agg_run writes them.  M: members (bagging: prob = raw / M); sum_a: Σ a_m (SAMME).
cudaError_t launch_agg_finalize(int kind, int C, int K, int dim, int loss, int M, double sum_a, int64_t n, int64_t ld,
                                float* raw, float* prob, float* label, int sms, cudaStream_t s);
cudaError_t launch_linear_predict(const float* X, int64_t n, int64_t ld, int n_coef,
                                  const float* coef, const int32_t* cols, float intercept,
                                  float* out, int sms, cudaStream_t s);

// ---- exact quantile by radix select (se_util.cu) ---------------------------------------------
// One pass: histogram (256 bins, fp64 counts in `hist`) of byte `shift/8` of the order-preserving key of each
// value whose higher bytes equal `prefix` (mask = bits above the byte).  value = a[i], or |a[i] - b[i]| when b.
cudaError_t launch_radix_hist(const float* a, const float* b, int64_t n, uint32_t prefix, uint32_t mask,
                              int shift, double* hist, int sms, cudaStream_t s);

// ---- ingest (se_util.cu): row-major host chunk [rows][d] -> column-major X[d][ld] rows [row0, row0+rows)
cudaError_t launch_transpose_rows(const float* src, int64_t rows, int d, float* X, int64_t ld, int64_t row0,
                                  cudaStream_t s);

// ---- utilities (se_util.cu) ------------------------------------------------------------------
// raises *bad (mapped host memory) when a label is not an integer class index in [0, K)
cudaError_t launch_validate_labels(const float* y, int64_t n, int K, int* bad, int sms, cudaStream_t s);
cudaError_t launch_fill(float* p, float v, int64_t n, int sms, cudaStream_t s);
cudaError_t launch_fill_synthetic(float* p, int kind, uint64_t seed, double a, double b, int64_t n,
                                  int64_t index_offset, int sms, cudaStream_t s);
cudaError_t launch_f64_to_f32(const double* src, float* dst, int64_t n, int sms, cudaStream_t s);
cudaError_t launch_scale_copy(const float* src, float* dst, float scale, int64_t n, int sms,
                              cudaStream_t s);

}  // namespace se
