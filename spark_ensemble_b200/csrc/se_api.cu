// se_api.cu — host side of libse_b200.so: the extern "C" ABI declared in include/se_abi.h.
//
// Owns the per-GPU context (stream, device slots, reduction workspace, scalar block, NCCL
// communicator) and turns each ABI call into kernel launches on the context stream.  No CPU
// fallback exists: every compute entry point needs a working CUDA device.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <sched.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/se_abi.h"
#define SE_BRENT_HOST_ONLY
#include "se_brent.h"
#include "se_kernels.h"
#include "se_loss.cuh"

using namespace se;

// ------------------------------------------------------------------------------------------------
// NCCL is bound at run time (dlopen) so the library loads on boxes/processes without it and never
// clashes with a copy another component (e.g. a host framework) already loaded.
// ------------------------------------------------------------------------------------------------
namespace {

typedef struct { char internal[128]; } nccl_uid_t;
typedef void* nccl_comm_t;
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(nccl_uid_t*) = nullptr;
  int (*CommInitRank)(nccl_comm_t*, int, nccl_uid_t, int) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  int (*GetVersion)(int*) = nullptr;
  bool ok = false;
  std::string why;
};
constexpr int kNcclFloat64 = 8;  // ncclDouble
constexpr int kNcclSum = 0;
constexpr int kNcclMax = 2;
constexpr int kNcclChar = 0;

void nccl_load(NcclApi& api);

NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] { nccl_load(api); });
  return api;
}

void nccl_load(NcclApi& api) {
  const char* names[] = {getenv("SE_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    if (!nm || !*nm) continue;
    api.handle = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
    if (api.handle) break;
  }
  if (!api.handle) {
    const char* de = dlerror();
    api.why = std::string("dlopen(libnccl.so.2) failed: ") + (de ? de : "?");
    return;
  }
#define SE_SYM(field, name)                                                     \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.handle, name));   \
  if (!api.field) { api.why = std::string("missing symbol ") + name; return; }
  SE_SYM(GetUniqueId, "ncclGetUniqueId")
  SE_SYM(CommInitRank, "ncclCommInitRank")
  SE_SYM(CommDestroy, "ncclCommDestroy")
  SE_SYM(AllReduce, "ncclAllReduce")
  SE_SYM(AllGather, "ncclAllGather")
  SE_SYM(GetErrorString, "ncclGetErrorString")
  SE_SYM(GetVersion, "ncclGetVersion")
#undef SE_SYM
  api.ok = true;
}

thread_local std::string g_last_error;

constexpr int kScal = 1024;         // doubles in the device/host scalar blocks ([0, 160): generic reductions)
constexpr int kScalHist = 704;      // 256-bin radix-select histogram
constexpr int kScalRound = 160;     // offset of the squared-round results (statistics, alpha, loss)
constexpr int64_t kL2HintRows = 16000000;  // 16 B/row of y, F, h, r: up to ~2x the 126 MB L2
constexpr int kScalHost = 192;      // offset used by se_comm_allreduce_host (up to kScalHist - kScalHost values)
constexpr int kSmallBytes = 1 << 20;  // small device scratch: weights, init, tree arrays, factors

struct SlotBuf {
  float* d = nullptr;
  int64_t rows = 0, cols = 0, ld = 0;
  size_t bytes = 0;
};

// uint8 rank matrix of a feature-matrix slot for the tree walk (se_models.cu): per column the sorted thresholds seen
// so far (<= 255), X8[col][i] = #{thresholds of col strictly below X[col][i]}
struct BinState {
  uint8_t* d8 = nullptr;
  int64_t ld8 = 0, n = 0;
  int d = 0;
  bool valid = false;                      // X8 reflects the current contents of the slot for every column with edges
  std::vector<std::vector<float>> edges;   // per column
  std::vector<char> dirty;
  float* d_edges = nullptr;                // [d][256]
  int32_t* d_nedges = nullptr;             // [d]
  int32_t* d_cols = nullptr;               // [d]
  uint4* d_nodes = nullptr;
  size_t nodes_cap = 0;
};

}  // namespace

struct se_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timing = false;
  double last_ms = 0.0;
  int sms = 148;
  int ctas_per_sm = 8;  // upper bound; launchers scale the grid down for small shards (se_gbm.cu grid_for)
  int64_t launches = 0;
  SlotBuf slot[SE_NUM_SLOTS];
  double* d_scal = nullptr;
  double* h_scal = nullptr;  // pinned
  double* d_partials = nullptr;
  unsigned int* d_counter = nullptr;
  unsigned char* d_small = nullptr;
  unsigned char* h_small = nullptr;  // pinned staging for d_small
  float* h_stage = nullptr;          // pinned staging for f64 uploads / scaled downloads
  size_t h_stage_bytes = 0;
  struct {
    bool on = false;
    int64_t n = 0, nv = 0;
    int dim = 1, loss = 0;
    double param = 0.0;
    bool has_w = false;
    bool use_bag = false;
    bool r_current = false;  // SE_SLOT_R holds -g(y, F) of the CURRENT F (squared loss: y - F)
    double wsum = 0.0;
    bool wsum_valid = false;
    double n_global = 0.0, nv_global = 0.0;
    bool counts_valid = false;
  } gbm;
  struct {
    bool on = false;
    int64_t n = 0;
    int K = 2;
    bool real = false;
  } boost;
  struct {
    bool on = false;
    int kind = 0, M = 0, K = 0, dim = 1, loss = 0, width = 1, C = 1;
    int64_t n = 0;
  } agg;
  struct {
    bool on = false;
    int64_t n = 0;
  } boostreg;
  nccl_comm_t comm = nullptr;
  int nranks = 1, rank = 0;
  // fused NVLink all-reduce: mailboxes of all ranks mapped into this process with CUDA IPC
  bool p2p = false;
  double* mbox_local = nullptr;
  std::vector<void*> mbox_peers;      // opened IPC mappings (index = rank; own entry = mbox_local)
  std::vector<char> mbox_ipc;         // 1: mbox_peers[p] came from cudaIpcOpenMemHandle (close it); 0: same-process peer pointer
  double** d_mbox_table = nullptr;    // device copy of the pointer table
  int* d_p2p_err = nullptr;           // device alias of h_p2p_err (mapped pinned host memory: no copy to poll it)
  int* h_p2p_err = nullptr;
  int* h_bad_label = nullptr;         // raised by kernels that met a label / vote outside [0, K) (mapped pinned memory)
  int* d_bad_label = nullptr;
  // labels used as class indices are validated once per upload: 0 unknown, 1 validation launched (result not yet
  // observed), 2 known good — per label slot (SE_SLOT_Y, SE_SLOT_VY) together with the K they were checked for
  int y_state[2] = {0, 0};
  int y_state_k[2] = {0, 0};
  unsigned long long red_seq = 0;
  bool last_reduce_global = false;    // the kernel just launched already produced cross-GPU sums
  // host mirror of the scalar block (mapped pinned memory written by the reducing kernel's last CTA)
  double* h_mirror = nullptr;         // [kMboxPayload] + ticket word
  double* d_mirror = nullptr;         // device alias
  unsigned long long mirror_ticket = 0;
  bool mirror_valid = false;
  int mirror_off = 0;
  bool use_mirror = true;
  float* d_ls_u = nullptr;            // line-search view (signed): u = (2y-1)F, v = (2y-1)h
  float* d_ls_v = nullptr;
  int64_t ls_cap = 0;
  bool ls_packed = false;             // evaluations currently read (u, v) instead of (y, F, h)
  unsigned pass_parity = 0;           // alternates the tile direction of consecutive GBM passes (L2 reuse)
  bool alternate = true;
  int l2_hints = -1;                  // evict_first hints on the GBM streams: -1 by shard size, 0 off, 1 on (SE_L2_HINTS)
  // ---- cooperative whole-round / whole-line-search kernels (se_gbm_fused.cu)
  FusedSync* d_fsync = nullptr;
  unsigned long long fused_epoch = 0;
  int fused_round = -1;               // squared-loss round in one launch: -1 by shard size, 0 off, 1 on
  int64_t fused_round_max_rows = (int64_t)1 << 40;  // measured faster than two launches from 6 M to 100 M rows
  int fused_ctas_per_sm = 3;
  double fused_prefetch_mb = 0.0;     // (measured: no gain at 6-12 M rows, -2 % at 25-50 M rows: off)
  int fused_loss_reduce = 0;          // 1: reduce the train loss over the rows even when the closed form applies
  int fused_l2_mode = 0;              // experiment: 1 = evict_last on r/h, 2 = persisting window over r
  int fused_timing = 0;               // diagnostic: in-kernel %globaltimer stamps of the fused round
  double last_fused_us[3] = {0, 0, 0};  // statistics phase, fold+exchange+Brent, update phase    // L2 budget of the update-phase prefetch issued while the grid waits for the step
  int ls_mode = 1;                    // non-squared line search: 0 one launch per evaluation (round-1 kernels), 1 one
                                      // persistent launch (device Brent), 2 host Brent over single-evaluation launches of
                                      // the persistent kernel (bit-identity check of mode 1)
  int ls_resident = 1;                // workers keep their first tiles in shared memory
  int ls_ctas_per_sm = 4;
  int ls_ring = 0;                    // cp.async ring stages for the streamed tiles (0 off = register prefetch, 2..4; measured: no gain)
  int l2_persist = 0;                 // mark the packed line-search view as L2-persisting.  OFF by default: measured on
                                      // B200 the 83 MB carve-out buys the search nothing (2.86 vs 2.75 ms of evaluations per
                                      // round at 50 M rows) and, while it is configured, every STREAMING kernel runs 2x slower
                                      // (K1 0.36 vs 0.17 ms at 50 M rows) — profiles/r02_ls_sweep.json
  size_t l2_persist_max = 0;          // cudaDevAttrMaxPersistingL2CacheSize
  size_t l2_window_max = 0;           // cudaDevAttrMaxAccessPolicyWindowSize
  size_t l2_persist_set = 0;          // current cudaLimitPersistingL2CacheSize
  double l2_persist_frac = 0.75;      // fraction of the persisting carve-out the window is sized for
  bool l2_persist_dirty = false;      // persisting lines may be resident: reset before unrelated kernels
  int clock_khz = 1965000;
  double peer_timeout_ms = 120000.0;  // spin bound of the fused peer exchange (0 = wait forever)
  // diagnostics of the last call (se_ctx_get_option)
  int last_round_fused = 0, last_ls_workers = 0, last_ls_resident = 0, last_ls_passes = 0, last_fused_grid = 0;
  double last_ls_hit_ratio = 0.0;
  double last_round_stats[3] = {0.0, 0.0, 0.0};
  // newton updates: SE_SLOT_WOUT holds 1/2 hc w; the 1/S_j of each dimension is applied on download
  std::vector<float> wout_scale;
  bool wout_scaled = false;
  // LogLoss with more than kMaxDim classes (se_gbm_generic.cu): buffers sized for the configured dim
  struct {
    int dim = 0, grid = 0;
    float* d_coef = nullptr;
    float* h_coef = nullptr;      // pinned
    double* d_partials = nullptr; // [grid][dim + 1]
    double* d_out = nullptr;      // [dim + 1]
    double* h_out = nullptr;      // pinned
    bool pending = false;         // the last GBM launch left its sums in d_out
  } big;
  // binned (uint8) copies of X / VX for the tree walk
  BinState bins[2];
  int tree_bins = 1;                  // 0: always walk the fp32 matrix
  unsigned char* d_forest = nullptr;  // packed chunk of trees for se_forest_predict / se_forest_classify
  size_t forest_cap = 0;
  float* d_forest_leaves = nullptr;   // leaf table of se_forest_classify (every tree's leaves, one or K floats each)
  size_t forest_leaves_cap = 0;
  int last_forest_chunks = 0;
  int wm_fast = 1;                    // weighted median (M <= 64, weights >= 0): keys-only sort + margin check, exact kernel for the rest
  int64_t wm_list_cap = 0;            // deferred-row list capacity (0: n / 4)
  unsigned int* d_wm = nullptr;       // [0] deferred count, [1..] row list
  size_t wm_alloc = 0;                // entries allocated in d_wm (count included)
  int last_wm_mode = 0;
  int tree_mask = 1;                  // shallow trees (<= 64 internal nodes): all-nodes comparison kernel over the rank matrix
  int last_tree_mask = 0;
  int last_tree_binned = 0, last_tree_rebinned_cols = 0;
  std::string err;
  // stopwatch + per-kernel-family timing
  cudaEvent_t tm0 = nullptr, tm1 = nullptr;
  bool ktiming = false;
  static constexpr int kRing = 128;
  cudaEvent_t kev[kRing][2] = {};
  int kfam[kRing] = {};
  int kpending = 0;
  double kms[SE_KF_COUNT] = {};
  int64_t kcount[SE_KF_COUNT] = {};
};

namespace {

int fail(se_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (ctx) ctx->err = buf;
  return code;
}

#define SE_CUDA(ctx, call)                                                                    \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(ctx, SE_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,              \
                  cudaGetErrorString(e__));                                                   \
  } while (0)

#define SE_LAUNCH(ctx, call)                                                                  \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    (ctx)->launches++;                                                                        \
    if (e__ != cudaSuccess)                                                                   \
      return fail(ctx, SE_ERR_CUDA, "%s:%d launch %s -> %s", __FILE__, __LINE__, #call,       \
                  cudaGetErrorString(e__));                                                   \
  } while (0)

int drain_kernel_events(se_ctx* ctx) {
  if (ctx->kpending == 0) return SE_OK;
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < ctx->kpending; ++i) {
    float ms = 0.f;
    SE_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->kev[i][0], ctx->kev[i][1]));
    ctx->kms[ctx->kfam[i]] += (double)ms;
    ctx->kcount[ctx->kfam[i]] += 1;
  }
  ctx->kpending = 0;
  return SE_OK;
}

// launch bracketed by CUDA events on the context stream when kernel timing is on
#define SE_LAUNCH_T(ctx, family, call)                                                        \
  do {                                                                                        \
    int slot__ = -1;                                                                          \
    if ((ctx)->ktiming) {                                                                     \
      if ((ctx)->kpending == se_ctx::kRing) {                                                 \
        int rc__ = drain_kernel_events(ctx);                                                  \
        if (rc__ != SE_OK) return rc__;                                                       \
      }                                                                                       \
      slot__ = (ctx)->kpending;                                                               \
      if (!(ctx)->kev[slot__][0]) {                                                           \
        SE_CUDA(ctx, cudaEventCreate(&(ctx)->kev[slot__][0]));                                \
        SE_CUDA(ctx, cudaEventCreate(&(ctx)->kev[slot__][1]));                                \
      }                                                                                       \
      SE_CUDA(ctx, cudaEventRecord((ctx)->kev[slot__][0], (ctx)->stream));                    \
    }                                                                                         \
    SE_LAUNCH(ctx, call);                                                                     \
    if (slot__ >= 0) {                                                                        \
      SE_CUDA(ctx, cudaEventRecord((ctx)->kev[slot__][1], (ctx)->stream));                    \
      (ctx)->kfam[slot__] = (family);                                                         \
      (ctx)->kpending = slot__ + 1;                                                           \
    }                                                                                         \
  } while (0)

#define SE_TRY(expr)                \
  do {                              \
    int rc__ = (expr);              \
    if (rc__ != SE_OK) return rc__; \
  } while (0)

#define SE_REQUIRE(ctx, cond, code, ...) \
  do {                                   \
    if (!(cond)) return fail(ctx, code, __VA_ARGS__); \
  } while (0)

// A non-sticky error left behind by an unrelated earlier runtime call (e.g. a query that reported "not ready")
// must not be mistaken for a failure of the next kernel launch, which is checked with cudaGetLastError().
void clear_stale_error(const char* where) {
  const cudaError_t stale = cudaGetLastError();
  if (stale != cudaSuccess && getenv("SE_DEBUG"))
    fprintf(stderr, "[se_b200] cleared stale CUDA error at %s: %s\n", where, cudaGetErrorString(stale));
}

int begin(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  clear_stale_error("begin");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->timing) SE_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  return SE_OK;
}

int end(se_ctx* ctx) {
  if (ctx->timing) SE_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  if (getenv("SE_DEBUG")) clear_stale_error("end");
  return SE_OK;
}

// exchange = true: the launched kernel ends in block_reduce_publish/peer_exchange (sum); it then performs
// the cross-GPU reduction itself over peer memory and the NCCL all-reduce is skipped.
RedWs red_ws(se_ctx* ctx, int out_offset = 0, bool exchange = true) {
  RedWs ws;
  ws.partials = ctx->d_partials;
  ws.counter = ctx->d_counter;
  ws.out = ctx->d_scal + out_offset;
  ws.bad_label = ctx->d_bad_label;
  ctx->last_reduce_global = false;
  ctx->mirror_valid = false;
  // results can be mirrored to the host by the kernel itself when they are final on this GPU: single GPU, or
  // the fused peer exchange (with the NCCL fallback the all-reduce still has to run after the kernel)
  if (exchange && ctx->use_mirror && ctx->h_mirror && (ctx->nranks <= 1 || ctx->p2p)) {
    ws.host_out = ctx->d_mirror;
    ws.host_flag = reinterpret_cast<volatile unsigned long long*>(ctx->d_mirror + kMboxPayload);
    ws.host_ticket = ++ctx->mirror_ticket;
    ctx->mirror_valid = true;
    ctx->mirror_off = out_offset;
  }
  if (exchange && ctx->p2p && ctx->nranks > 1) {
    ws.mbox = ctx->d_mbox_table;
    ws.nranks = ctx->nranks;
    ws.rank = ctx->rank;
    ws.seq = ++ctx->red_seq;
    ws.err = ctx->d_p2p_err;
    ws.timeout_clocks = (long long)(ctx->peer_timeout_ms * (double)ctx->clock_khz);
    ctx->last_reduce_global = true;
  }
  return ws;
}

// all-reduce d_scal[off..off+count) in-stream (no-op without communicator)
int allreduce_dev(se_ctx* ctx, int off, int count, int op = kNcclSum) {
  if (!ctx->comm || ctx->nranks <= 1) return SE_OK;
  if (ctx->last_reduce_global && op == kNcclSum) {  // already summed across GPUs inside the kernel
    ctx->last_reduce_global = false;
    return SE_OK;
  }
  NcclApi& api = nccl();
  int rc = api.AllReduce(ctx->d_scal + off, ctx->d_scal + off, (size_t)count, kNcclFloat64, op,
                         ctx->comm, ctx->stream);
  if (rc != 0) return fail(ctx, SE_ERR_NCCL, "ncclAllReduce: %s", api.GetErrorString(rc));
  return SE_OK;
}

// Labels are class indices for LogLoss / SAMME(.R) / vote aggregation.  The reference throws on the JVM for a label
// outside [0, numClasses) or a fractional one (GBMLoss.scala:200-204 `res(label.toInt) = 1.0`, Classifier.validateLabel);
// here the kernels raise a flag instead of indexing out of bounds and the call that observes it fails with SE_ERR_ARG.
int check_labels(se_ctx* ctx) {
  if (!(ctx->h_bad_label && *reinterpret_cast<volatile int*>(ctx->h_bad_label))) {
    for (int& st : ctx->y_state)
      if (st == 1) st = 2;  // a validation pass completed before this point (same stream) and raised nothing
    return SE_OK;
  }
  if (ctx->h_bad_label) {
    ctx->y_state[0] = ctx->y_state[1] = 0;  // unknown again: the next call re-validates (and fails again if unchanged)
    *reinterpret_cast<volatile int*>(ctx->h_bad_label) = 0;
    return fail(ctx, SE_ERR_ARG, "a label (or vote) is not an integer class index in [0, numClasses): results of this call are invalid");
  }
  return SE_OK;
}

int check_p2p(se_ctx* ctx) {
  if (ctx->p2p && ctx->h_p2p_err && *reinterpret_cast<volatile int*>(ctx->h_p2p_err))
    return fail(ctx, SE_ERR_NCCL, "peer-memory all-reduce failed: a rank did not launch the matching reduction within "
                "%.0f ms (or gave up on it); se_comm_clear_error() re-arms the communicator", ctx->peer_timeout_ms);
  return SE_OK;
}

// Wait until the kernel's last CTA has written the current mirror ticket into mapped host memory.  Spins on the
// cache line with PAUSE for the first ~100 us (the common case: the kernel is already running), then yields the core
// between polls so that a long kernel / a slow peer does not burn the driver thread.
int wait_mirror(se_ctx* ctx) {
  volatile unsigned long long* flag = reinterpret_cast<volatile unsigned long long*>(ctx->h_mirror + kMboxPayload);
  for (unsigned long spin = 0;; ++spin) {
    if (*flag == ctx->mirror_ticket) return SE_OK;
    if (spin < 20000) {
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
      continue;
    }
    if ((spin & 0x3F) == 0) {
      const cudaError_t q = cudaStreamQuery(ctx->stream);
      if (q != cudaErrorNotReady) {  // finished or failed
        if (*flag == ctx->mirror_ticket) return SE_OK;
        if (q != cudaSuccess) return fail(ctx, SE_ERR_CUDA, "kernel failed before publishing its results: %s", cudaGetErrorString(q));
        SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (*flag == ctx->mirror_ticket) return SE_OK;
        return fail(ctx, SE_ERR_CUDA, "reduction results never reached the host mirror");
      }
    }
    sched_yield();
  }
}

// (all-reduce and) bring d_scal[off..off+count) to the host; synchronises the stream
int fetch_scalars(se_ctx* ctx, int off, int count, double* out, int op = kNcclSum) {
  if (ctx->mirror_valid && ctx->mirror_off == off && op == kNcclSum && count <= kMboxPayload) {
    // poll the ticket the last CTA writes after the sums: no D2H copy, no stream synchronisation
    ctx->mirror_valid = false;
    ctx->last_reduce_global = false;
    SE_TRY(end(ctx));
    SE_TRY(wait_mirror(ctx));
    for (int i = 0; i < count; ++i) out[i] = ctx->h_mirror[i];
    SE_TRY(check_labels(ctx));
    return check_p2p(ctx);
  }
  SE_TRY(allreduce_dev(ctx, off, count, op));
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + off, ctx->d_scal + off, sizeof(double) * count,
                               cudaMemcpyDeviceToHost, ctx->stream));
  SE_TRY(end(ctx));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < count; ++i) out[i] = ctx->h_scal[off + i];
  SE_TRY(check_labels(ctx));
  return check_p2p(ctx);
}

// any write to a feature-matrix slot makes its rank matrix stale
void touch_slot(se_ctx* ctx, int slot) {
  if (slot == SE_SLOT_Y) ctx->y_state[0] = 0;
  if (slot == SE_SLOT_VY) ctx->y_state[1] = 0;
  if (slot == SE_SLOT_WOUT) ctx->wout_scaled = false;
  if (slot == SE_SLOT_X) ctx->bins[0].valid = false;
  if (slot == SE_SLOT_VX) ctx->bins[1].valid = false;
}

void free_bins(BinState& B) {
  if (B.d8) cudaFree(B.d8);
  if (B.d_edges) cudaFree(B.d_edges);
  if (B.d_nedges) cudaFree(B.d_nedges);
  if (B.d_cols) cudaFree(B.d_cols);
  if (B.d_nodes) cudaFree(B.d_nodes);
  B = BinState();
}

int slot_alloc2d(se_ctx* ctx, int slot, int64_t rows, int64_t cols) {
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  SE_REQUIRE(ctx, rows >= 1 && cols >= 0, SE_ERR_ARG, "bad slot shape %lld x %lld", (long long)rows,
             (long long)cols);
  SlotBuf& s = ctx->slot[slot];
  const int64_t ld = (rows > 1) ? ((cols + 31) / 32) * 32 : cols;
  const size_t bytes = sizeof(float) * (size_t)(rows * ld + 32);
  if (s.d && s.bytes >= bytes) {
    s.rows = rows; s.cols = cols; s.ld = ld;
    return SE_OK;
  }
  if (s.d) SE_CUDA(ctx, cudaFree(s.d));
  s = SlotBuf();
  SE_CUDA(ctx, cudaMalloc(&s.d, bytes));
  s.rows = rows; s.cols = cols; s.ld = ld; s.bytes = bytes;
  return SE_OK;
}

int need_slot(se_ctx* ctx, int slot, int64_t rows, int64_t cols, const char* what) {
  const SlotBuf& s = ctx->slot[slot];
  if (!s.d || s.rows != rows || s.cols != cols)
    return fail(ctx, SE_ERR_STATE, "%s: slot %d must hold [%lld][%lld] (has [%lld][%lld])", what,
                slot, (long long)rows, (long long)cols, (long long)s.rows, (long long)s.cols);
  return SE_OK;
}

int ensure_stage(se_ctx* ctx, size_t bytes) {
  if (ctx->h_stage_bytes >= bytes) return SE_OK;
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  ctx->h_stage = nullptr;
  ctx->h_stage_bytes = 0;
  SE_CUDA(ctx, cudaMallocHost(&ctx->h_stage, bytes));
  ctx->h_stage_bytes = bytes;
  return SE_OK;
}

// logical flat [rows][cols] range -> per-row physical segments
template <class Fn>
int for_segments(se_ctx* ctx, const SlotBuf& s, int64_t count, int64_t offset, Fn fn) {
  SE_REQUIRE(ctx, s.d, SE_ERR_STATE, "slot not allocated");
  SE_REQUIRE(ctx, offset >= 0 && count >= 0 && offset + count <= s.rows * s.cols, SE_ERR_ARG,
             "range [%lld,+%lld) outside slot of %lld elements", (long long)offset,
             (long long)count, (long long)(s.rows * s.cols));
  int64_t done = 0;
  while (done < count) {
    const int64_t pos = offset + done;
    const int64_t r = (s.cols > 0) ? pos / s.cols : 0, c = (s.cols > 0) ? pos % s.cols : 0;
    int64_t len = s.cols - c;
    if (len > count - done) len = count - done;
    SE_TRY(fn(s.d + r * s.ld + c, done, len));
    done += len;
  }
  return SE_OK;
}

// Release L2 lines a previous line search marked as persisting (they would otherwise keep occupying the carve-out
// while unrelated kernels stream through a smaller L2).
int release_l2_persist(se_ctx* ctx) {
  if (!ctx->l2_persist_dirty) return SE_OK;
  ctx->l2_persist_dirty = false;
  cudaCtxResetPersistingL2Cache();
  // the carve-out itself (not only the lines in it) slows streaming kernels down: give the L2 back
  cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
  ctx->l2_persist_set = 0;
  cudaGetLastError();
  return SE_OK;
}

int ensure_counts(se_ctx* ctx) {
  if (ctx->gbm.counts_valid) return SE_OK;
  SE_CUDA(ctx, cudaSetDevice(ctx->device));  // callers may run before begin(): launches below need the right device
  double v[2] = {(double)ctx->gbm.n, (double)ctx->gbm.nv};
  SE_TRY(se_comm_allreduce_host(ctx, v, 2));
  ctx->gbm.n_global = v[0];
  ctx->gbm.nv_global = v[1];
  ctx->gbm.counts_valid = true;
  return SE_OK;
}

int ensure_wsum(se_ctx* ctx) {
  if (ctx->gbm.wsum_valid) return SE_OK;
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_TRY(ensure_counts(ctx));
  if (ctx->gbm.use_bag) {
    // weightSum over the bag: Σ c_i·w_i (GBMLoss.scala:65 adds instance.weight once per sampled copy)
    SE_TRY(need_slot(ctx, SE_SLOT_BAG, 1, ctx->gbm.n, "bag multiplicities"));
    SE_LAUNCH(ctx, launch_dot(ctx->slot[SE_SLOT_BAG].d, ctx->gbm.has_w ? ctx->slot[SE_SLOT_W].d : nullptr,
                              ctx->gbm.n, red_ws(ctx), ctx->ctas_per_sm, ctx->sms, ctx->stream));
    double s = 0.0;
    SE_TRY(fetch_scalars(ctx, 0, 1, &s));
    ctx->gbm.wsum = s;
  } else if (!ctx->gbm.has_w) {
    ctx->gbm.wsum = ctx->gbm.n_global;
  } else {
    SE_TRY(need_slot(ctx, SE_SLOT_W, 1, ctx->gbm.n, "instance weights"));
    SE_LAUNCH(ctx, launch_sum(ctx->slot[SE_SLOT_W].d, ctx->gbm.n, red_ws(ctx), ctx->ctas_per_sm,
                              ctx->sms, ctx->stream));
    double s = 0.0;
    SE_TRY(fetch_scalars(ctx, 0, 1, &s));
    ctx->gbm.wsum = s;
  }
  ctx->gbm.wsum_valid = true;
  return SE_OK;
}

GbmArgs gbm_args(se_ctx* ctx, bool validation) {
  GbmArgs a;
  const auto& g = ctx->gbm;
  a.y = ctx->slot[validation ? SE_SLOT_VY : SE_SLOT_Y].d;
  a.F = ctx->slot[validation ? SE_SLOT_VF : SE_SLOT_F].d;
  a.h = ctx->slot[validation ? SE_SLOT_VH : SE_SLOT_H].d;
  a.w = (!validation && g.has_w) ? ctx->slot[SE_SLOT_W].d : nullptr;
  a.bag = (!validation && g.use_bag) ? ctx->slot[SE_SLOT_BAG].d : nullptr;
  a.r = validation ? nullptr : ctx->slot[SE_SLOT_R].d;
  a.wout = validation ? nullptr : ctx->slot[SE_SLOT_WOUT].d;
  a.n = validation ? g.nv : g.n;
  a.ld = ctx->slot[validation ? SE_SLOT_VF : SE_SLOT_F].ld;
  a.dim = g.dim;
  a.param = (float)g.param;
  a.reverse = (ctx->alternate && !validation) ? (int)(ctx->pass_parity++ & 1u) : 0;
  // shards whose four per-row arrays (y, F, h, r) are of the order of the L2: evict_first hints (se_common.cuh)
  a.l2_hints = ctx->l2_hints >= 0 ? ctx->l2_hints : ((validation ? ctx->gbm.nv : ctx->gbm.n) <= kL2HintRows ? 1 : 0);
  a.ws = red_ws(ctx, 0, /*exchange=*/false);  // armed (sequence number taken) only at reducing launches
  return a;
}

// ---- Brent (se_brent.h): host wrapper over the shared host/device template
int brent_impl(se_fn1 f, void* user, double lo, double hi, double start, double rel, double abs_tol,
               int max_eval, double* x_out, double* f_out, int* n_eval) {
  const int rc = brent_core([&](double x) { return f(x, user); }, lo, hi, start, rel, abs_tol, max_eval, x_out, f_out,
                            n_eval);
  return rc == kBrentOk ? SE_OK : SE_ERR_OPT;
}

}  // namespace

// ================================================================================================
extern "C" {

int se_abi_version(void) { return SE_ABI_VERSION; }

const char* se_last_error(const se_ctx* ctx) {
  if (ctx && !ctx->err.empty()) return ctx->err.c_str();
  return g_last_error.c_str();
}

int se_device_count(int* out) {
  if (!out) return fail(nullptr, SE_ERR_ARG, "null out");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    *out = 0;
    return fail(nullptr, SE_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  *out = n;
  return SE_OK;
}

int se_ctx_create(int device, se_ctx** out) {
  if (!out) return fail(nullptr, SE_ERR_ARG, "null out");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(nullptr, SE_ERR_CUDA, "no CUDA device available (%s): the hot path has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(nullptr, SE_ERR_ARG, "device %d out of range [0,%d)", device, n);
  se_ctx* ctx = new se_ctx();
  ctx->device = device;
#define SE_CREATE_CUDA(call)                                                            \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      int rc__ = fail(nullptr, SE_ERR_CUDA, "%s -> %s", #call, cudaGetErrorString(e__)); \
      delete ctx;                                                                       \
      return rc__;                                                                      \
    }                                                                                   \
  } while (0)
  SE_CREATE_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SE_CREATE_CUDA(cudaGetDeviceProperties(&prop, device));
  ctx->sms = prop.multiProcessorCount;
  if (const char* s = getenv("SE_ALTERNATE_PASSES")) ctx->alternate = atoi(s) != 0;
  if (const char* s = getenv("SE_L2_HINTS")) ctx->l2_hints = atoi(s) != 0 ? 1 : 0;
  if (const char* s = getenv("SE_CTAS_PER_SM")) {
    const int v = atoi(s);
    if (v >= 1 && v <= 16) ctx->ctas_per_sm = v;
  }
  SE_CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  SE_CREATE_CUDA(cudaEventCreate(&ctx->ev0));
  SE_CREATE_CUDA(cudaEventCreate(&ctx->ev1));
  SE_CREATE_CUDA(cudaMalloc(&ctx->d_scal, sizeof(double) * kScal));
  SE_CREATE_CUDA(cudaMemset(ctx->d_scal, 0, sizeof(double) * kScal));
  SE_CREATE_CUDA(cudaMallocHost(&ctx->h_scal, sizeof(double) * kScal));
  SE_CREATE_CUDA(cudaMalloc(&ctx->d_partials, sizeof(double) * (size_t)kMaxGridPartials * kMaxRed));
  SE_CREATE_CUDA(cudaMalloc(&ctx->d_counter, sizeof(unsigned int)));
  SE_CREATE_CUDA(cudaMemset(ctx->d_counter, 0, sizeof(unsigned int)));
  SE_CREATE_CUDA(cudaHostAlloc(&ctx->h_bad_label, sizeof(int), cudaHostAllocMapped));
  *ctx->h_bad_label = 0;
  SE_CREATE_CUDA(cudaHostGetDevicePointer(&ctx->d_bad_label, ctx->h_bad_label, 0));
  SE_CREATE_CUDA(cudaMalloc(&ctx->d_fsync, sizeof(FusedSync)));
  SE_CREATE_CUDA(cudaMemset(ctx->d_fsync, 0, sizeof(FusedSync)));
  ctx->clock_khz = prop.clockRate > 0 ? prop.clockRate : 1965000;
  {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxPersistingL2CacheSize, device) == cudaSuccess && v > 0) ctx->l2_persist_max = (size_t)v;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxAccessPolicyWindowSize, device) == cudaSuccess && v > 0) ctx->l2_window_max = (size_t)v;
    cudaGetLastError();
  }
  if (const char* s = getenv("SE_FUSED_ROUND")) ctx->fused_round = atoi(s) != 0 ? 1 : 0;
  if (const char* s = getenv("SE_LS_MODE")) { const int v = atoi(s); if (v >= 0 && v <= 2) ctx->ls_mode = v; }
  if (const char* s = getenv("SE_LS_RESIDENT")) ctx->ls_resident = atoi(s) != 0;
  if (const char* s = getenv("SE_LS_RING")) { const int v = atoi(s); if (v >= 0 && v <= 4) ctx->ls_ring = v; }
  if (const char* s = getenv("SE_L2_PERSIST")) ctx->l2_persist = atoi(s) != 0;
  if (const char* s = getenv("SE_PEER_TIMEOUT_MS")) { const double v = atof(s); if (v >= 0.0) ctx->peer_timeout_ms = v; }
  SE_CREATE_CUDA(cudaHostAlloc(&ctx->h_mirror, sizeof(double) * (kMboxPayload + 8), cudaHostAllocMapped));
  memset(ctx->h_mirror, 0, sizeof(double) * (kMboxPayload + 8));
  SE_CREATE_CUDA(cudaHostGetDevicePointer(&ctx->d_mirror, ctx->h_mirror, 0));
  if (const char* s = getenv("SE_HOST_MIRROR")) ctx->use_mirror = atoi(s) != 0;
  SE_CREATE_CUDA(cudaMalloc(&ctx->d_small, kSmallBytes));
  SE_CREATE_CUDA(cudaMallocHost(&ctx->h_small, kSmallBytes));
  SE_CREATE_CUDA(cudaDeviceSynchronize());
#undef SE_CREATE_CUDA
  *out = ctx;
  return SE_OK;
}

int se_ctx_destroy(se_ctx* ctx) {
  if (!ctx) return SE_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->comm && nccl().ok) {
    for (int p = 0; p < (int)ctx->mbox_peers.size(); ++p)
      if (p != ctx->rank && ctx->mbox_peers[p] && ctx->mbox_ipc[p]) cudaIpcCloseMemHandle(ctx->mbox_peers[p]);
    if (ctx->mbox_local) cudaFree(ctx->mbox_local);
    if (ctx->d_mbox_table) cudaFree(ctx->d_mbox_table);
    if (ctx->h_p2p_err) cudaFreeHost(ctx->h_p2p_err);
    nccl().CommDestroy(ctx->comm);
  }
  for (auto& s : ctx->slot)
    if (s.d) cudaFree(s.d);
  if (ctx->d_scal) cudaFree(ctx->d_scal);
  if (ctx->h_scal) cudaFreeHost(ctx->h_scal);
  if (ctx->d_partials) cudaFree(ctx->d_partials);
  if (ctx->d_counter) cudaFree(ctx->d_counter);
  if (ctx->d_fsync) cudaFree(ctx->d_fsync);
  free_bins(ctx->bins[0]);
  free_bins(ctx->bins[1]);
  if (ctx->d_wm) cudaFree(ctx->d_wm);
  if (ctx->d_forest) cudaFree(ctx->d_forest);
  if (ctx->d_forest_leaves) cudaFree(ctx->d_forest_leaves);
  if (ctx->big.d_coef) cudaFree(ctx->big.d_coef);
  if (ctx->big.h_coef) cudaFreeHost(ctx->big.h_coef);
  if (ctx->big.d_partials) cudaFree(ctx->big.d_partials);
  if (ctx->big.d_out) cudaFree(ctx->big.d_out);
  if (ctx->big.h_out) cudaFreeHost(ctx->big.h_out);
  if (ctx->h_bad_label) cudaFreeHost(ctx->h_bad_label);
  if (ctx->d_small) cudaFree(ctx->d_small);
  if (ctx->h_mirror) cudaFreeHost(ctx->h_mirror);
  if (ctx->d_ls_u) cudaFree(ctx->d_ls_u);  // (u, v) share one allocation
  if (ctx->h_small) cudaFreeHost(ctx->h_small);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->tm0) cudaEventDestroy(ctx->tm0);
  if (ctx->tm1) cudaEventDestroy(ctx->tm1);
  for (auto& pr : ctx->kev) { if (pr[0]) cudaEventDestroy(pr[0]); if (pr[1]) cudaEventDestroy(pr[1]); }
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return SE_OK;
}

int se_ctx_sync(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return check_labels(ctx);
}

int se_ctx_device(const se_ctx* ctx, int* device) {
  if (!ctx || !device) return fail(nullptr, SE_ERR_ARG, "null argument");
  *device = ctx->device;
  return SE_OK;
}

int se_ctx_launch_count(const se_ctx* ctx, int64_t* out) {
  if (!ctx || !out) return fail(nullptr, SE_ERR_ARG, "null argument");
  *out = ctx->launches;
  return SE_OK;
}

int se_ctx_set_timing(se_ctx* ctx, int on) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  ctx->timing = on != 0;
  return SE_OK;
}

int se_ctx_last_ms(se_ctx* ctx, double* out) {
  if (!ctx || !out) return fail(nullptr, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->timing, SE_ERR_STATE, "timing is off (se_ctx_set_timing)");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  float ms = 0.f;
  SE_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  *out = (double)ms;
  return SE_OK;
}

int se_ctx_timer_start(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!ctx->tm0) {
    SE_CUDA(ctx, cudaEventCreate(&ctx->tm0));
    SE_CUDA(ctx, cudaEventCreate(&ctx->tm1));
  }
  SE_CUDA(ctx, cudaEventRecord(ctx->tm0, ctx->stream));
  return SE_OK;
}

int se_ctx_timer_stop(se_ctx* ctx, double* ms) {
  if (!ctx || !ms) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->tm0, SE_ERR_STATE, "se_ctx_timer_start first");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaEventRecord(ctx->tm1, ctx->stream));
  SE_CUDA(ctx, cudaEventSynchronize(ctx->tm1));
  float f = 0.f;
  SE_CUDA(ctx, cudaEventElapsedTime(&f, ctx->tm0, ctx->tm1));
  *ms = (double)f;
  return SE_OK;
}

int se_ctx_kernel_timing(se_ctx* ctx, int on) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!on) SE_TRY(drain_kernel_events(ctx));
  ctx->ktiming = on != 0;
  return SE_OK;
}

int se_ctx_kernel_time(se_ctx* ctx, int family, double* total_ms, int64_t* launches) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, family >= 0 && family < SE_KF_COUNT, SE_ERR_ARG, "bad kernel family %d", family);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_TRY(drain_kernel_events(ctx));
  if (total_ms) *total_ms = ctx->kms[family];
  if (launches) *launches = ctx->kcount[family];
  return SE_OK;
}

int se_ctx_kernel_time_reset(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_TRY(drain_kernel_events(ctx));
  for (int i = 0; i < SE_KF_COUNT; ++i) { ctx->kms[i] = 0.0; ctx->kcount[i] = 0; }
  return SE_OK;
}

namespace {
struct OptKey { const char* name; int id; };
enum { OPT_LAST_FOREST_CHUNKS, OPT_WM_FAST, OPT_WM_LIST_CAP, OPT_LAST_WM_MODE, OPT_LAST_WM_DEFERRED, OPT_TREE_MASK, OPT_LAST_TREE_MASK, OPT_TREE_BINS, OPT_LAST_TREE_BINNED, OPT_LAST_TREE_REBINNED, OPT_FUSED_LOSS_REDUCE, OPT_FUSED_L2_MODE, OPT_FUSED_TIMING, OPT_LAST_FUSED_US0, OPT_LAST_FUSED_US1, OPT_LAST_FUSED_US2, OPT_FUSED_PREFETCH_MB, OPT_FUSED_ROUND, OPT_FUSED_MAX_ROWS, OPT_FUSED_CTAS, OPT_LS_MODE, OPT_LS_RESIDENT, OPT_LS_CTAS, OPT_LS_RING, OPT_L2_PERSIST,
       OPT_L2_PERSIST_FRAC, OPT_PEER_TIMEOUT_MS, OPT_ALTERNATE, OPT_L2_HINTS, OPT_CTAS_PER_SM, OPT_HOST_MIRROR,
       // read-only diagnostics
       OPT_LAST_ROUND_FUSED, OPT_LAST_LS_WORKERS, OPT_LAST_LS_PASSES, OPT_LAST_LS_HIT_RATIO, OPT_LAST_FUSED_GRID,
       OPT_L2_PERSIST_MAX, OPT_L2_WINDOW_MAX, OPT_LAST_STAT0, OPT_LAST_STAT1, OPT_LAST_STAT2 };
const OptKey kOpts[] = {
  {"last_forest_chunks", OPT_LAST_FOREST_CHUNKS}, {"wm_fast", OPT_WM_FAST}, {"wm_list_cap", OPT_WM_LIST_CAP}, {"last_wm_mode", OPT_LAST_WM_MODE}, {"last_wm_deferred", OPT_LAST_WM_DEFERRED},
  {"tree_bins", OPT_TREE_BINS}, {"tree_mask", OPT_TREE_MASK}, {"last_tree_mask", OPT_LAST_TREE_MASK}, {"last_tree_binned", OPT_LAST_TREE_BINNED}, {"last_tree_rebinned_cols", OPT_LAST_TREE_REBINNED},
  {"fused_loss_reduce", OPT_FUSED_LOSS_REDUCE}, {"fused_l2_mode", OPT_FUSED_L2_MODE}, {"fused_timing", OPT_FUSED_TIMING}, {"last_fused_stats_us", OPT_LAST_FUSED_US0}, {"last_fused_brent_us", OPT_LAST_FUSED_US1},
  {"last_fused_update_us", OPT_LAST_FUSED_US2}, {"fused_prefetch_mb", OPT_FUSED_PREFETCH_MB}, {"fused_round", OPT_FUSED_ROUND}, {"fused_round_max_rows", OPT_FUSED_MAX_ROWS}, {"fused_ctas_per_sm", OPT_FUSED_CTAS},
  {"ls_mode", OPT_LS_MODE}, {"ls_resident", OPT_LS_RESIDENT}, {"ls_ctas_per_sm", OPT_LS_CTAS}, {"ls_ring", OPT_LS_RING}, {"l2_persist", OPT_L2_PERSIST},
  {"l2_persist_frac", OPT_L2_PERSIST_FRAC}, {"peer_timeout_ms", OPT_PEER_TIMEOUT_MS}, {"alternate_passes", OPT_ALTERNATE},
  {"l2_hints", OPT_L2_HINTS}, {"ctas_per_sm", OPT_CTAS_PER_SM}, {"host_mirror", OPT_HOST_MIRROR},
  {"last_round_fused", OPT_LAST_ROUND_FUSED}, {"last_ls_workers", OPT_LAST_LS_WORKERS}, {"last_ls_passes", OPT_LAST_LS_PASSES},
  {"last_ls_hit_ratio", OPT_LAST_LS_HIT_RATIO}, {"last_fused_grid", OPT_LAST_FUSED_GRID},
  {"l2_persist_max_bytes", OPT_L2_PERSIST_MAX}, {"l2_window_max_bytes", OPT_L2_WINDOW_MAX},
  {"last_round_stat0", OPT_LAST_STAT0}, {"last_round_stat1", OPT_LAST_STAT1}, {"last_round_stat2", OPT_LAST_STAT2},
};
int opt_id(const char* key) {
  if (!key) return -1;
  for (const OptKey& k : kOpts)
    if (strcmp(k.name, key) == 0) return k.id;
  return -1;
}
}  // namespace

int se_ctx_set_option(se_ctx* ctx, const char* key, double value) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  const int iv = (int)value;
  switch (opt_id(key)) {
    case OPT_FUSED_ROUND: ctx->fused_round = value < 0 ? -1 : (iv != 0); break;
    case OPT_FUSED_MAX_ROWS: ctx->fused_round_max_rows = (int64_t)value; break;
    case OPT_FUSED_TIMING: ctx->fused_timing = iv != 0; break;
    case OPT_FUSED_LOSS_REDUCE: ctx->fused_loss_reduce = iv != 0; break;
    case OPT_TREE_BINS: ctx->tree_bins = iv != 0; break;
    case OPT_TREE_MASK: ctx->tree_mask = iv != 0; break;
    case OPT_WM_FAST: ctx->wm_fast = iv != 0; break;
    case OPT_WM_LIST_CAP: SE_REQUIRE(ctx, value >= 0 && value < 2147483000.0, SE_ERR_ARG, "wm_list_cap in [0, 2^31)"); ctx->wm_list_cap = (int64_t)value; break;
    case OPT_FUSED_L2_MODE: SE_REQUIRE(ctx, iv >= 0 && iv <= 2, SE_ERR_ARG, "fused_l2_mode in {0,1,2}"); ctx->fused_l2_mode = iv; if (iv != 2) release_l2_persist(ctx); break;
    case OPT_FUSED_PREFETCH_MB: SE_REQUIRE(ctx, value >= 0.0 && value <= 512.0, SE_ERR_ARG, "fused_prefetch_mb in [0,512]"); ctx->fused_prefetch_mb = value; break;
    case OPT_FUSED_CTAS: SE_REQUIRE(ctx, iv >= 1 && iv <= 8, SE_ERR_ARG, "fused_ctas_per_sm in [1,8]"); ctx->fused_ctas_per_sm = iv; break;
    case OPT_LS_MODE: SE_REQUIRE(ctx, iv >= 0 && iv <= 2, SE_ERR_ARG, "ls_mode in {0,1,2}"); ctx->ls_mode = iv; break;
    case OPT_LS_RESIDENT: ctx->ls_resident = iv != 0; break;
    case OPT_LS_RING: SE_REQUIRE(ctx, iv >= 0 && iv <= 4, SE_ERR_ARG, "ls_ring in [0,4]"); ctx->ls_ring = iv; break;
    case OPT_LS_CTAS: SE_REQUIRE(ctx, iv >= 1 && iv <= 8, SE_ERR_ARG, "ls_ctas_per_sm in [1,8]"); ctx->ls_ctas_per_sm = iv; break;
    case OPT_L2_PERSIST: ctx->l2_persist = iv != 0; break;
    case OPT_L2_PERSIST_FRAC: SE_REQUIRE(ctx, value > 0.0 && value <= 1.0, SE_ERR_ARG, "l2_persist_frac in (0,1]"); ctx->l2_persist_frac = value; break;
    case OPT_PEER_TIMEOUT_MS: SE_REQUIRE(ctx, value >= 0.0, SE_ERR_ARG, "peer_timeout_ms >= 0"); ctx->peer_timeout_ms = value; break;
    case OPT_ALTERNATE: ctx->alternate = iv != 0; break;
    case OPT_L2_HINTS: ctx->l2_hints = value < 0 ? -1 : (iv != 0); break;
    case OPT_CTAS_PER_SM: SE_REQUIRE(ctx, iv >= 1 && iv <= 16, SE_ERR_ARG, "ctas_per_sm in [1,16]"); ctx->ctas_per_sm = iv; break;
    case OPT_HOST_MIRROR: ctx->use_mirror = iv != 0; break;
    default: return fail(ctx, SE_ERR_ARG, "unknown or read-only option '%s'", key ? key : "(null)");
  }
  return SE_OK;
}

int se_ctx_get_option(const se_ctx* ctx, const char* key, double* value) {
  if (!ctx || !value) return fail(nullptr, SE_ERR_ARG, "null argument");
  switch (opt_id(key)) {
    case OPT_FUSED_ROUND: *value = ctx->fused_round; break;
    case OPT_FUSED_MAX_ROWS: *value = (double)ctx->fused_round_max_rows; break;
    case OPT_FUSED_PREFETCH_MB: *value = ctx->fused_prefetch_mb; break;
    case OPT_FUSED_TIMING: *value = ctx->fused_timing; break;
    case OPT_FUSED_LOSS_REDUCE: *value = ctx->fused_loss_reduce; break;
    case OPT_TREE_BINS: *value = ctx->tree_bins; break;
    case OPT_TREE_MASK: *value = ctx->tree_mask; break;
    case OPT_WM_FAST: *value = ctx->wm_fast; break;
    case OPT_LAST_FOREST_CHUNKS: *value = ctx->last_forest_chunks; break;
    case OPT_WM_LIST_CAP: *value = (double)ctx->wm_list_cap; break;
    case OPT_LAST_WM_MODE: *value = ctx->last_wm_mode; break;
    case OPT_LAST_WM_DEFERRED: {  // rows the last weighted median sent to the exact kernel (synchronises the stream)
      unsigned int c = 0;
      if (ctx->d_wm && ctx->last_wm_mode == 1) {
        cudaSetDevice(ctx->device);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || cudaMemcpy(&c, ctx->d_wm, sizeof(c), cudaMemcpyDeviceToHost) != cudaSuccess) {
          cudaGetLastError();
          return SE_ERR_CUDA;
        }
      }
      *value = (double)c;
      break;
    }
    case OPT_LAST_TREE_MASK: *value = ctx->last_tree_mask; break;
    case OPT_LAST_TREE_BINNED: *value = ctx->last_tree_binned; break;
    case OPT_LAST_TREE_REBINNED: *value = ctx->last_tree_rebinned_cols; break;
    case OPT_FUSED_L2_MODE: *value = ctx->fused_l2_mode; break;
    case OPT_LAST_FUSED_US0: *value = ctx->last_fused_us[0]; break;
    case OPT_LAST_FUSED_US1: *value = ctx->last_fused_us[1]; break;
    case OPT_LAST_FUSED_US2: *value = ctx->last_fused_us[2]; break;
    case OPT_FUSED_CTAS: *value = ctx->fused_ctas_per_sm; break;
    case OPT_LS_MODE: *value = ctx->ls_mode; break;
    case OPT_LS_RESIDENT: *value = ctx->ls_resident; break;
    case OPT_LS_RING: *value = ctx->ls_ring; break;
    case OPT_LS_CTAS: *value = ctx->ls_ctas_per_sm; break;
    case OPT_L2_PERSIST: *value = ctx->l2_persist; break;
    case OPT_L2_PERSIST_FRAC: *value = ctx->l2_persist_frac; break;
    case OPT_PEER_TIMEOUT_MS: *value = ctx->peer_timeout_ms; break;
    case OPT_ALTERNATE: *value = ctx->alternate; break;
    case OPT_L2_HINTS: *value = ctx->l2_hints; break;
    case OPT_CTAS_PER_SM: *value = ctx->ctas_per_sm; break;
    case OPT_HOST_MIRROR: *value = ctx->use_mirror; break;
    case OPT_LAST_ROUND_FUSED: *value = ctx->last_round_fused; break;
    case OPT_LAST_LS_WORKERS: *value = ctx->last_ls_workers; break;
    case OPT_LAST_LS_PASSES: *value = ctx->last_ls_passes; break;
    case OPT_LAST_LS_HIT_RATIO: *value = ctx->last_ls_hit_ratio; break;
    case OPT_LAST_FUSED_GRID: *value = ctx->last_fused_grid; break;
    case OPT_L2_PERSIST_MAX: *value = (double)ctx->l2_persist_max; break;
    case OPT_L2_WINDOW_MAX: *value = (double)ctx->l2_window_max; break;
    case OPT_LAST_STAT0: *value = ctx->last_round_stats[0]; break;
    case OPT_LAST_STAT1: *value = ctx->last_round_stats[1]; break;
    case OPT_LAST_STAT2: *value = ctx->last_round_stats[2]; break;
    default: return fail(const_cast<se_ctx*>(ctx), SE_ERR_ARG, "unknown option '%s'", key ? key : "(null)");
  }
  return SE_OK;
}

int se_host_alloc(int64_t bytes, void** out) {
  if (!out || bytes < 0) return fail(nullptr, SE_ERR_ARG, "bad argument");
  *out = nullptr;
  cudaError_t e = cudaMallocHost(out, (size_t)(bytes > 0 ? bytes : 1));
  if (e != cudaSuccess) return fail(nullptr, SE_ERR_CUDA, "cudaMallocHost(%lld): %s", (long long)bytes, cudaGetErrorString(e));
  return SE_OK;
}

int se_host_free(void* ptr) {
  if (!ptr) return SE_OK;
  cudaError_t e = cudaFreeHost(ptr);
  if (e != cudaSuccess) return fail(nullptr, SE_ERR_CUDA, "cudaFreeHost: %s", cudaGetErrorString(e));
  return SE_OK;
}

// ---- communicator ------------------------------------------------------------------------------
int se_comm_unique_id(void* out, int bytes) {
  if (!out || bytes < SE_COMM_ID_BYTES) return fail(nullptr, SE_ERR_ARG, "id buffer must hold %d bytes", SE_COMM_ID_BYTES);
  NcclApi& api = nccl();
  if (!api.ok) return fail(nullptr, SE_ERR_NCCL, "NCCL unavailable: %s", api.why.c_str());
  nccl_uid_t id;
  int rc = api.GetUniqueId(&id);
  if (rc != 0) return fail(nullptr, SE_ERR_NCCL, "ncclGetUniqueId: %s", api.GetErrorString(rc));
  memcpy(out, &id, sizeof(id));
  return SE_OK;
}

int se_comm_init(se_ctx* ctx, int nranks, int rank, const void* id, int bytes) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, nranks >= 1 && rank >= 0 && rank < nranks, SE_ERR_ARG, "bad rank %d of %d", rank, nranks);
  SE_REQUIRE(ctx, !ctx->comm, SE_ERR_STATE, "communicator already attached");
  ctx->nranks = nranks;
  ctx->rank = rank;
  ctx->gbm.counts_valid = ctx->gbm.wsum_valid = false;
  if (nranks == 1) return SE_OK;
  SE_REQUIRE(ctx, id && bytes >= SE_COMM_ID_BYTES, SE_ERR_ARG, "unique id of %d bytes required", SE_COMM_ID_BYTES);
  NcclApi& api = nccl();
  if (!api.ok) return fail(ctx, SE_ERR_NCCL, "NCCL unavailable: %s", api.why.c_str());
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  nccl_uid_t uid;
  memcpy(&uid, id, sizeof(uid));
  int rc = api.CommInitRank(&ctx->comm, nranks, uid, rank);
  if (rc != 0) {
    ctx->comm = nullptr;
    return fail(ctx, SE_ERR_NCCL, "ncclCommInitRank: %s", api.GetErrorString(rc));
  }
  // ---- peer-memory mailboxes for the fused all-reduce (falls back to NCCL if any rank cannot map them)
  const char* env = getenv("SE_P2P_ALLREDUCE");
  int want = (env && atoi(env) == 0) ? 0 : 1;
  const size_t mbox_bytes = sizeof(double) * (size_t)nranks * 2 * kMboxStride;
  int ok = want;
  cudaIpcMemHandle_t mine;
  memset(&mine, 0, sizeof(mine));
  if (ok) {
    ok = cudaMalloc(&ctx->mbox_local, mbox_bytes) == cudaSuccess && cudaMemset(ctx->mbox_local, 0, mbox_bytes) == cudaSuccess &&
         cudaHostAlloc(&ctx->h_p2p_err, sizeof(int), cudaHostAllocMapped) == cudaSuccess &&
         cudaHostGetDevicePointer(&ctx->d_p2p_err, ctx->h_p2p_err, 0) == cudaSuccess &&
         cudaMalloc(&ctx->d_mbox_table, sizeof(double*) * nranks) == cudaSuccess &&
         cudaIpcGetMemHandle(&mine, ctx->mbox_local) == cudaSuccess;
    cudaGetLastError();
  }
  // exchange the handles (and everyone's readiness) through NCCL.  Ranks that live in the SAME process (one JVM /
  // one Python process driving several GPUs: sharded.ShardedContext) cannot open each other's IPC handles — they
  // exchange the raw device pointer instead and enable peer access between the two devices.
  struct PeerBlob { cudaIpcMemHandle_t handle; unsigned char ok; unsigned char pad[3]; int32_t pid; int32_t device; int32_t pad2; uint64_t ptr; };
  const size_t hb = sizeof(PeerBlob);
  std::vector<unsigned char> send(hb, 0), recv(hb * nranks, 0);
  {
    PeerBlob b;
    memset(&b, 0, sizeof(b));
    b.handle = mine; b.ok = (unsigned char)ok; b.pid = (int32_t)getpid(); b.device = ctx->device;
    b.ptr = (uint64_t)(uintptr_t)ctx->mbox_local;
    memcpy(send.data(), &b, sizeof(b));
  }
  unsigned char *d_send = nullptr, *d_recv = nullptr;
  SE_CUDA(ctx, cudaMalloc(&d_send, hb));
  SE_CUDA(ctx, cudaMalloc(&d_recv, hb * nranks));
  SE_CUDA(ctx, cudaMemcpyAsync(d_send, send.data(), hb, cudaMemcpyHostToDevice, ctx->stream));
  rc = api.AllGather(d_send, d_recv, hb, kNcclChar, ctx->comm, ctx->stream);
  if (rc != 0) {
    cudaFree(d_send);
    cudaFree(d_recv);
    return fail(ctx, SE_ERR_NCCL, "ncclAllGather: %s", api.GetErrorString(rc));
  }
  SE_CUDA(ctx, cudaMemcpyAsync(recv.data(), d_recv, hb * nranks, cudaMemcpyDeviceToHost, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int all_ok = 1;
  for (int p = 0; p < nranks; ++p) all_ok &= reinterpret_cast<const PeerBlob*>(recv.data() + p * hb)->ok;
  ctx->mbox_peers.assign(nranks, nullptr);
  ctx->mbox_ipc.assign(nranks, 0);
  if (all_ok) {
    for (int p = 0; p < nranks && all_ok; ++p) {
      if (p == rank) { ctx->mbox_peers[p] = ctx->mbox_local; continue; }
      PeerBlob b;
      memcpy(&b, recv.data() + p * hb, sizeof(b));
      void* ptr = nullptr;
      if (b.pid == (int32_t)getpid()) {
        int can = 0;
        if (b.device == ctx->device) can = 1;
        else if (cudaDeviceCanAccessPeer(&can, ctx->device, b.device) == cudaSuccess && can) {
          const cudaError_t pe = cudaDeviceEnablePeerAccess(b.device, 0);
          if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) can = 0;
        }
        cudaGetLastError();
        if (can) ptr = (void*)(uintptr_t)b.ptr; else all_ok = 0;
      } else {
        if (cudaIpcOpenMemHandle(&ptr, b.handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { all_ok = 0; cudaGetLastError(); }
        else ctx->mbox_ipc[p] = 1;
      }
      ctx->mbox_peers[p] = ptr;
    }
  }
  // second round: did every rank manage to open every peer?
  send[0] = (unsigned char)all_ok;
  SE_CUDA(ctx, cudaMemcpyAsync(d_send, send.data(), hb, cudaMemcpyHostToDevice, ctx->stream));
  rc = api.AllGather(d_send, d_recv, hb, kNcclChar, ctx->comm, ctx->stream);
  if (rc != 0) return fail(ctx, SE_ERR_NCCL, "ncclAllGather: %s", api.GetErrorString(rc));
  SE_CUDA(ctx, cudaMemcpyAsync(recv.data(), d_recv, hb * nranks, cudaMemcpyDeviceToHost, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int p = 0; p < nranks; ++p) all_ok &= recv[p * hb];
  cudaFree(d_send);
  cudaFree(d_recv);
  if (all_ok) {
    *ctx->h_p2p_err = 0;
    SE_CUDA(ctx, cudaMemcpy(ctx->d_mbox_table, ctx->mbox_peers.data(), sizeof(double*) * nranks, cudaMemcpyHostToDevice));
    ctx->p2p = true;
    ctx->red_seq = 0;
  } else {
    ctx->p2p = false;  // NCCL all-reduce of the scalar block after each reducing kernel
  }
  return SE_OK;
}

int se_comm_p2p_active(const se_ctx* ctx, int* active) {
  if (!ctx || !active) return fail(nullptr, SE_ERR_ARG, "null argument");
  *active = ctx->p2p ? 1 : 0;
  return SE_OK;
}

int se_comm_clear_error(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->h_p2p_err) *reinterpret_cast<volatile int*>(ctx->h_p2p_err) = 0;
  ctx->err.clear();
  return SE_OK;
}

static void release_p2p(se_ctx* ctx) {
  for (int p = 0; p < (int)ctx->mbox_peers.size(); ++p)
    if (p != ctx->rank && ctx->mbox_peers[p] && ctx->mbox_ipc[p]) cudaIpcCloseMemHandle(ctx->mbox_peers[p]);
  ctx->mbox_peers.clear();
  ctx->mbox_ipc.clear();
  if (ctx->mbox_local) cudaFree(ctx->mbox_local);
  if (ctx->d_mbox_table) cudaFree(ctx->d_mbox_table);
  if (ctx->h_p2p_err) cudaFreeHost(ctx->h_p2p_err);
  ctx->mbox_local = nullptr; ctx->d_mbox_table = nullptr; ctx->d_p2p_err = nullptr; ctx->h_p2p_err = nullptr;
  ctx->p2p = false;
}

int se_comm_destroy(se_ctx* ctx) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  if (ctx->comm) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    release_p2p(ctx);
    nccl().CommDestroy(ctx->comm);
    ctx->comm = nullptr;
  }
  ctx->nranks = 1;
  ctx->rank = 0;
  ctx->gbm.counts_valid = ctx->gbm.wsum_valid = false;
  return SE_OK;
}

int se_comm_info(const se_ctx* ctx, int* nranks, int* rank) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  if (nranks) *nranks = ctx->nranks;
  if (rank) *rank = ctx->rank;
  return SE_OK;
}

int se_comm_allreduce_host(se_ctx* ctx, double* values, int count) {
  if (!ctx || !values) return fail(nullptr, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, count >= 0 && count <= kScalHist - kScalHost, SE_ERR_ARG, "count %d too large", count);
  if (!ctx->comm || ctx->nranks <= 1 || count == 0) return SE_OK;
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  for (int i = 0; i < count; ++i) ctx->h_scal[kScalHost + i] = values[i];
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_scal + kScalHost, ctx->h_scal + kScalHost, sizeof(double) * count,
                               cudaMemcpyHostToDevice, ctx->stream));
  ctx->last_reduce_global = false;
  SE_TRY(allreduce_dev(ctx, kScalHost, count));
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + kScalHost, ctx->d_scal + kScalHost, sizeof(double) * count,
                               cudaMemcpyDeviceToHost, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < count; ++i) values[i] = ctx->h_scal[kScalHost + i];
  return SE_OK;
}

// ---- slots -------------------------------------------------------------------------------------
int se_slot_alloc(se_ctx* ctx, int slot, int64_t count) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  return slot_alloc2d(ctx, slot, 1, count);
}

int se_slot_alloc2d(se_ctx* ctx, int slot, int64_t rows, int64_t cols) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  return slot_alloc2d(ctx, slot, rows, cols);
}

int se_slot_free(se_ctx* ctx, int slot) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->slot[slot].d) SE_CUDA(ctx, cudaFree(ctx->slot[slot].d));
  ctx->slot[slot] = SlotBuf();
  if (slot == SE_SLOT_X) free_bins(ctx->bins[0]);
  if (slot == SE_SLOT_VX) free_bins(ctx->bins[1]);
  return SE_OK;
}

int se_slot_info(const se_ctx* ctx, int slot, void** device_ptr, int64_t* count) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  if (slot < 0 || slot >= SE_NUM_SLOTS) return fail(nullptr, SE_ERR_ARG, "bad slot %d", slot);
  if (device_ptr) {
    *device_ptr = ctx->slot[slot].d;
    touch_slot(const_cast<se_ctx*>(ctx), slot);
    // the caller may write through the raw pointer: drop everything cached about the slot's contents
    se_ctx* mctx = const_cast<se_ctx*>(ctx);
    if (slot == SE_SLOT_Y || slot == SE_SLOT_F || slot == SE_SLOT_R) mctx->gbm.r_current = false;
    if (slot == SE_SLOT_W || slot == SE_SLOT_BAG) mctx->gbm.wsum_valid = false;
  }
  if (count) *count = ctx->slot[slot].rows * ctx->slot[slot].cols;
  return SE_OK;
}

int se_slot_layout(const se_ctx* ctx, int slot, int64_t* rows, int64_t* cols, int64_t* ld) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  if (slot < 0 || slot >= SE_NUM_SLOTS) return fail(nullptr, SE_ERR_ARG, "bad slot %d", slot);
  if (rows) *rows = ctx->slot[slot].rows;
  if (cols) *cols = ctx->slot[slot].cols;
  if (ld) *ld = ctx->slot[slot].ld;
  return SE_OK;
}

int se_upload(se_ctx* ctx, int slot, const float* host, int64_t count, int64_t offset) {
  if (!ctx || !host) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (slot == SE_SLOT_W || slot == SE_SLOT_BAG) ctx->gbm.wsum_valid = false;
  if (slot == SE_SLOT_Y || slot == SE_SLOT_F || slot == SE_SLOT_R) ctx->gbm.r_current = false;
  SE_TRY(for_segments(ctx, ctx->slot[slot], count, offset, [&](float* d, int64_t done, int64_t len) {
    SE_CUDA(ctx, cudaMemcpyAsync(d, host + done, sizeof(float) * len, cudaMemcpyHostToDevice, ctx->stream));
    return SE_OK;
  }));
  // host buffers are borrowed for the duration of the call only
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return SE_OK;
}

int se_upload_f64(se_ctx* ctx, int slot, const double* host, int64_t count, int64_t offset) {
  if (!ctx || !host) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (slot == SE_SLOT_W || slot == SE_SLOT_BAG) ctx->gbm.wsum_valid = false;
  if (slot == SE_SLOT_Y || slot == SE_SLOT_F || slot == SE_SLOT_R) ctx->gbm.r_current = false;
  // narrow on the host (halves PCIe bytes) through pinned staging, in chunks
  const int64_t chunk = 1 << 22;
  SE_TRY(ensure_stage(ctx, sizeof(float) * (size_t)chunk));
  SE_TRY(for_segments(ctx, ctx->slot[slot], count, offset, [&](float* d, int64_t done, int64_t len) {
    for (int64_t c0 = 0; c0 < len; c0 += chunk) {
      const int64_t m = (len - c0 < chunk) ? len - c0 : chunk;
      for (int64_t i = 0; i < m; ++i) ctx->h_stage[i] = (float)host[done + c0 + i];
      SE_CUDA(ctx, cudaMemcpyAsync(d + c0, ctx->h_stage, sizeof(float) * m, cudaMemcpyHostToDevice, ctx->stream));
      SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SE_OK;
  }));
  return SE_OK;
}

int se_upload_rowmajor(se_ctx* ctx, int slot, const float* host, int64_t n_rows, int d, int64_t row_offset) {
  if (!ctx || (!host && n_rows > 0)) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  const SlotBuf& X = ctx->slot[slot];
  SE_REQUIRE(ctx, X.d && X.rows == d, SE_ERR_STATE, "slot %d must be allocated as [%d][n] (has [%lld][%lld])", slot, d,
             (long long)X.rows, (long long)X.cols);
  SE_REQUIRE(ctx, n_rows >= 0 && row_offset >= 0 && row_offset + n_rows <= X.cols, SE_ERR_ARG,
             "rows [%lld,+%lld) outside the slot's %lld rows", (long long)row_offset, (long long)n_rows, (long long)X.cols);
  if (n_rows == 0) return SE_OK;
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t ld = X.rows > 1 ? X.ld : X.cols;
  // ~32 MB chunks, whole rows, multiple of 32 rows
  int64_t chunk_rows = (int64_t)(32u << 20) / ((int64_t)d * (int64_t)sizeof(float));
  chunk_rows = (chunk_rows / 32) * 32;
  if (chunk_rows < 32) chunk_rows = 32;
  if (chunk_rows > n_rows) chunk_rows = n_rows;
  const size_t chunk_bytes = (size_t)chunk_rows * d * sizeof(float);
  cudaPointerAttributes attr;
  const bool pinned_src = (cudaPointerGetAttributes(&attr, host) == cudaSuccess && attr.type == cudaMemoryTypeHost);
  cudaGetLastError();
  float* dstage[2] = {nullptr, nullptr};
  float* hstage[2] = {nullptr, nullptr};
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copied[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
  int rc = SE_OK;
  auto cleanup = [&]() {
    if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 2; ++i) {
      if (dstage[i]) cudaFree(dstage[i]);
      if (hstage[i]) cudaFreeHost(hstage[i]);
      if (copied[i]) cudaEventDestroy(copied[i]);
      if (consumed[i]) cudaEventDestroy(consumed[i]);
    }
  };
#define SE_ING(call)                                                                            \
  do {                                                                                          \
    cudaError_t e__ = (call);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      rc = fail(ctx, SE_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      cleanup();                                                                                \
      return rc;                                                                                \
    }                                                                                           \
  } while (0)
  SE_ING(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    SE_ING(cudaMalloc(&dstage[i], chunk_bytes));
    if (!pinned_src) SE_ING(cudaMallocHost(&hstage[i], chunk_bytes));
    SE_ING(cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming));
    SE_ING(cudaEventCreateWithFlags(&consumed[i], cudaEventDisableTiming));
  }
  int64_t done = 0;
  for (int c = 0; done < n_rows; ++c) {
    const int b = c & 1;
    const int64_t rows = (n_rows - done < chunk_rows) ? n_rows - done : chunk_rows;
    const size_t bytes = (size_t)rows * d * sizeof(float);
    if (c >= 2) SE_ING(cudaEventSynchronize(consumed[b]));  // staging buffers of chunk c-2 are free again
    const float* src = host + done * d;
    if (!pinned_src) {
      memcpy(hstage[b], src, bytes);  // overlaps the DMA of chunk c-1 and the transpose of chunk c-2
      src = hstage[b];
    }
    SE_ING(cudaMemcpyAsync(dstage[b], src, bytes, cudaMemcpyHostToDevice, copy_stream));
    SE_ING(cudaEventRecord(copied[b], copy_stream));
    SE_ING(cudaStreamWaitEvent(ctx->stream, copied[b], 0));
    cudaError_t le = launch_transpose_rows(dstage[b], rows, d, X.d, ld, row_offset + done, ctx->stream);
    ctx->launches++;
    if (le != cudaSuccess) SE_ING(le);
    SE_ING(cudaEventRecord(consumed[b], ctx->stream));
    done += rows;
  }
#undef SE_ING
  cleanup();
  return SE_OK;
}

int se_download(se_ctx* ctx, int slot, float* host, int64_t count, int64_t offset) {
  if (!ctx || !host) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_TRY(for_segments(ctx, ctx->slot[slot], count, offset, [&](float* d, int64_t done, int64_t len) {
    SE_CUDA(ctx, cudaMemcpyAsync(host + done, d, sizeof(float) * len, cudaMemcpyDeviceToHost, ctx->stream));
    return SE_OK;
  }));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (slot == SE_SLOT_WOUT && ctx->wout_scaled) {
    // newton base-learner weights: 1/2 hc w on the device, x 1/S_dim here (GBMRegressor.scala:379)
    const int64_t cols = ctx->slot[slot].cols;
    for (int64_t i = 0; i < count; ++i) {
      const size_t j = (size_t)(cols > 0 ? (offset + i) / cols : 0);
      if (j < ctx->wout_scale.size()) host[i] *= ctx->wout_scale[j];
    }
  }
  return check_labels(ctx);  // e.g. the probabilities of an aggregation that met a vote outside [0, K)
}

int se_download_scaled(se_ctx* ctx, int slot, double scale, float* host, int64_t count, int64_t offset) {
  if (!ctx || !host) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_TRY(se_download(ctx, slot, host, count, offset));
  const float s = (float)scale;
  for (int64_t i = 0; i < count; ++i) host[i] *= s;
  return SE_OK;
}

int se_fill(se_ctx* ctx, int slot, float value, int64_t count, int64_t offset) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (slot == SE_SLOT_W || slot == SE_SLOT_BAG) ctx->gbm.wsum_valid = false;
  if (slot == SE_SLOT_Y || slot == SE_SLOT_F || slot == SE_SLOT_R) ctx->gbm.r_current = false;
  return for_segments(ctx, ctx->slot[slot], count, offset, [&](float* d, int64_t, int64_t len) {
    SE_LAUNCH(ctx, launch_fill(d, value, len, ctx->sms, ctx->stream));
    return SE_OK;
  });
}

int se_copy_slot(se_ctx* ctx, int dst_slot, int src_slot) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, dst_slot >= 0 && dst_slot < SE_NUM_SLOTS && src_slot >= 0 && src_slot < SE_NUM_SLOTS,
             SE_ERR_ARG, "bad slot");
  const SlotBuf &d = ctx->slot[dst_slot], &s = ctx->slot[src_slot];
  SE_REQUIRE(ctx, d.d && s.d && d.rows == s.rows && d.cols == s.cols, SE_ERR_STATE, "slot shapes differ");
  touch_slot(ctx, dst_slot);
  if (dst_slot == SE_SLOT_Y || dst_slot == SE_SLOT_F || dst_slot == SE_SLOT_R) ctx->gbm.r_current = false;
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaMemcpyAsync(d.d, s.d, sizeof(float) * (size_t)(s.rows * s.ld), cudaMemcpyDeviceToDevice, ctx->stream));
  return SE_OK;
}

int se_fill_synthetic(se_ctx* ctx, int slot, int kind, uint64_t seed, double a, double b, int64_t count,
                      int64_t offset) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  touch_slot(ctx, slot);
  SE_REQUIRE(ctx, kind >= 0 && kind <= 3, SE_ERR_ARG, "bad synthetic kind %d", kind);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (slot == SE_SLOT_W || slot == SE_SLOT_BAG) ctx->gbm.wsum_valid = false;
  if (slot == SE_SLOT_Y || slot == SE_SLOT_F || slot == SE_SLOT_R) ctx->gbm.r_current = false;
  return for_segments(ctx, ctx->slot[slot], count, offset, [&](float* d, int64_t done, int64_t len) {
    SE_LAUNCH(ctx, launch_fill_synthetic(d, kind, seed, a, b, len, offset + done, ctx->sms, ctx->stream));
    return SE_OK;
  });
}

int se_slot_sum(se_ctx* ctx, int slot, int64_t count, double* out) {
  if (!ctx || !out) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
  const SlotBuf& s = ctx->slot[slot];
  SE_REQUIRE(ctx, s.d && s.rows == 1 && count <= s.cols, SE_ERR_STATE, "slot %d is not a [n] vector of >= %lld", slot, (long long)count);
  SE_TRY(begin(ctx));
  SE_LAUNCH(ctx, launch_sum(s.d, count, red_ws(ctx), ctx->ctas_per_sm, ctx->sms, ctx->stream));
  return fetch_scalars(ctx, 0, 1, out);
}

int se_quantile(se_ctx* ctx, int which, int slot, int64_t count, double q, double* out) {
  if (!ctx || !out) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, q >= 0.0 && q <= 1.0, SE_ERR_ARG, "quantile %g outside [0,1]", q);
  const float *a = nullptr, *b = nullptr;
  int64_t n = count;
  if (which == 1) {
    SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.dim == 1, SE_ERR_STATE, "|y - F| quantile needs a dim-1 GBM problem");
    a = ctx->slot[SE_SLOT_Y].d;
    b = ctx->slot[SE_SLOT_F].d;
    n = ctx->gbm.n;
  } else {
    SE_REQUIRE(ctx, slot >= 0 && slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad slot %d", slot);
    const SlotBuf& s = ctx->slot[slot];
    SE_REQUIRE(ctx, s.d && s.rows == 1 && count <= s.cols, SE_ERR_STATE, "slot %d is not a [n] vector of >= %lld", slot, (long long)count);
    a = s.d;
  }
  SE_TRY(begin(ctx));
  double total = (double)n;
  SE_TRY(se_comm_allreduce_host(ctx, &total, 1));
  SE_REQUIRE(ctx, total >= 1.0, SE_ERR_ARG, "quantile of an empty column");
  // 1-based target rank: ceil(q·N), at least 1
  double rank = ceil(q * total);
  if (rank < 1.0) rank = 1.0;
  uint32_t prefix = 0, mask = 0;
  double hist[256];
  for (int shift = 24; shift >= 0; shift -= 8) {
    SE_CUDA(ctx, cudaMemsetAsync(ctx->d_scal + kScalHist, 0, sizeof(double) * 256, ctx->stream));
    ctx->last_reduce_global = false;  // histogram bins: summed by NCCL
    SE_LAUNCH_T(ctx, SE_KF_OTHER, launch_radix_hist(a, b, n, prefix, mask, shift, ctx->d_scal + kScalHist, ctx->sms, ctx->stream));
    SE_TRY(fetch_scalars(ctx, kScalHist, 256, hist));
    double cum = 0.0;
    int bin = 255;
    for (int i = 0; i < 256; ++i) {
      if (cum + hist[i] >= rank) { bin = i; break; }
      cum += hist[i];
    }
    rank -= cum;
    prefix |= (uint32_t)bin << shift;
    mask |= 0xFFu << shift;
  }
  // invert the order-preserving key
  const uint32_t bits = (prefix & 0x80000000u) ? (prefix & 0x7FFFFFFFu) : ~prefix;
  float v;
  memcpy(&v, &bits, sizeof(v));
  *out = (double)v;
  return SE_OK;
}

// ---- GBM ---------------------------------------------------------------------------------------
int se_gbm_configure(se_ctx* ctx, int64_t n_train, int64_t n_valid, int dim, int loss, double param,
                     int has_weights) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, n_train >= 0 && n_valid >= 0, SE_ERR_ARG, "negative row count");
  SE_REQUIRE(ctx, loss >= SE_LOSS_SQUARED && loss <= SE_LOSS_LOGLOSS, SE_ERR_ARG, "unknown loss %d", loss);
  SE_REQUIRE(ctx, dim >= 1 && dim <= kMaxDimGeneric, SE_ERR_ARG, "dim %d outside [1,%d]", dim, kMaxDimGeneric);
  SE_REQUIRE(ctx, (loss == SE_LOSS_LOGLOSS) || dim == 1, SE_ERR_ARG, "scalar losses have dim 1 (got %d)", dim);
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  auto& g = ctx->gbm;
  g.on = true; g.n = n_train; g.nv = n_valid; g.dim = dim; g.loss = loss; g.param = param;
  g.has_w = has_weights != 0;
  g.use_bag = false;
  g.r_current = false;
  g.wsum_valid = false; g.counts_valid = false;
  ctx->y_state[0] = ctx->y_state[1] = 0;
  release_l2_persist(ctx);
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_Y, 1, n_train));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_F, dim, n_train));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_H, dim, n_train));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_R, dim, n_train));
  if (g.has_w) SE_TRY(slot_alloc2d(ctx, SE_SLOT_W, 1, n_train));
  // validation slots exist even for an EMPTY local validation shard (trailing row shards may be empty,
  // ensemble.row_partition): the rank must still launch every validation reduction so that its peers' collectives complete
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_VY, 1, n_valid));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_VF, dim, n_valid));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_VH, dim, n_valid));
  return SE_OK;
}

int se_gbm_set_loss_param(se_ctx* ctx, double param) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  ctx->gbm.param = param;
  ctx->gbm.r_current = false;
  return SE_OK;
}

int se_gbm_set_bag(se_ctx* ctx, int on) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  if (on) SE_TRY(slot_alloc2d(ctx, SE_SLOT_BAG, 1, ctx->gbm.n));
  ctx->gbm.use_bag = on != 0;
  ctx->gbm.wsum_valid = false;
  return SE_OK;
}

namespace {
int ensure_big(se_ctx* ctx, int dim) {
  auto& b = ctx->big;
  if (b.dim >= dim && b.d_out) return SE_OK;
  if (b.d_coef) cudaFree(b.d_coef);
  if (b.h_coef) cudaFreeHost(b.h_coef);
  if (b.d_partials) cudaFree(b.d_partials);
  if (b.d_out) cudaFree(b.d_out);
  if (b.h_out) cudaFreeHost(b.h_out);
  b.d_coef = nullptr; b.h_coef = nullptr; b.d_partials = nullptr; b.d_out = nullptr; b.h_out = nullptr; b.dim = 0; b.grid = 0; b.pending = false;
  int grid = ctx->sms * 8;
  if (grid > 1024) grid = 1024;
  SE_CUDA(ctx, cudaMalloc(&b.d_coef, sizeof(float) * (size_t)dim));
  SE_CUDA(ctx, cudaMallocHost(&b.h_coef, sizeof(float) * (size_t)dim));
  SE_CUDA(ctx, cudaMalloc(&b.d_partials, sizeof(double) * (size_t)grid * (size_t)(dim + 1)));
  SE_CUDA(ctx, cudaMalloc(&b.d_out, sizeof(double) * (size_t)(dim + 1)));
  SE_CUDA(ctx, cudaMallocHost(&b.h_out, sizeof(double) * (size_t)(dim + 1)));
  b.dim = dim;
  b.grid = grid;
  return SE_OK;
}

// Labels as class indices: one validation pass per upload of the label slot (see validate_labels_kernel).
int ensure_labels_checked(se_ctx* ctx, int which /*0 train, 1 validation*/, int K, int64_t n) {
  if (ctx->y_state[which] == 2 && ctx->y_state_k[which] == K) return SE_OK;
  const SlotBuf& y = ctx->slot[which ? SE_SLOT_VY : SE_SLOT_Y];
  if (!y.d || n <= 0) return SE_OK;
  SE_LAUNCH(ctx, launch_validate_labels(y.d, n, K, ctx->d_bad_label, ctx->sms, ctx->stream));
  ctx->y_state[which] = 1;
  ctx->y_state_k[which] = K;
  return SE_OK;
}

// One GBM kernel launch for the configured loss.  `coef` (alpha or step, gbm.dim values, nullable) goes into the kernel
// arguments for dim <= kMaxDim and into a device buffer for the general LogLoss path beyond it.
int gbm_launch(se_ctx* ctx, int family, int mode, GbmArgs& a, const double* coef) {
  const int dim = ctx->gbm.dim;
  ctx->big.pending = false;
  if (ctx->gbm.loss == SE_LOSS_LOGLOSS) {
    const int which = (a.y == ctx->slot[SE_SLOT_VY].d && a.y != nullptr && a.y != ctx->slot[SE_SLOT_Y].d) ? 1 : 0;
    SE_TRY(ensure_labels_checked(ctx, which, dim, a.n));
  }
  if (dim <= kMaxDim) {
    if (coef)
      for (int j = 0; j < dim; ++j) a.coef[j] = (float)coef[j];
    SE_LAUNCH_T(ctx, family, launch_gbm(ctx->gbm.loss, mode, a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
    return SE_OK;
  }
  SE_TRY(ensure_big(ctx, dim));
  auto& b = ctx->big;
  if (coef) {
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // h_coef may still feed the previous launch
    for (int j = 0; j < dim; ++j) b.h_coef[j] = (float)coef[j];
    SE_CUDA(ctx, cudaMemcpyAsync(b.d_coef, b.h_coef, sizeof(float) * (size_t)dim, cudaMemcpyHostToDevice, ctx->stream));
  }
  GenericArgs ga;
  ga.coef = b.d_coef;
  ga.partials = b.d_partials;
  ga.out = b.d_out;
  const int64_t groups = (a.n + 31) / 32;
  int grid = (int)(groups < (int64_t)b.grid ? (groups > 0 ? groups : 1) : b.grid);
  // the sums of this path are all-reduced by NCCL (fetch below): disarm the in-kernel exchange / host mirror
  ctx->last_reduce_global = false;
  ctx->mirror_valid = false;
  SE_LAUNCH_T(ctx, family, launch_gbm_logloss_generic(mode, a, ga, grid, ctx->stream));
  b.pending = true;
  return SE_OK;
}

// The sums of the last gbm_launch: [0] Σloss, [1 + j] per-dimension sums — global (summed across GPUs).
int gbm_fetch(se_ctx* ctx, int count, double* out) {
  if (!ctx->big.pending) return fetch_scalars(ctx, 0, count, out);
  auto& b = ctx->big;
  b.pending = false;
  if (ctx->comm && ctx->nranks > 1) {
    NcclApi& api = nccl();
    int rc = api.AllReduce(b.d_out, b.d_out, (size_t)(ctx->gbm.dim + 1), kNcclFloat64, kNcclSum, ctx->comm, ctx->stream);
    if (rc != 0) return fail(ctx, SE_ERR_NCCL, "ncclAllReduce: %s", api.GetErrorString(rc));
  }
  SE_CUDA(ctx, cudaMemcpyAsync(b.h_out, b.d_out, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
  SE_TRY(end(ctx));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < count; ++i) out[i] = b.h_out[i];
  return check_labels(ctx);
}
}  // namespace

static int newton_finish(se_ctx* ctx, double* sum_hess) {
  // S_j (all-reduced) -> the base-learner weights are WOUT_j * 1/S_j  (GBMRegressor.scala:373,379;
  // GBMClassifier.scala:344-355,364).  The kernel left the unnormalised 1/2 hc w in SE_SLOT_WOUT; the per-dimension
  // factor 1/S_j is applied where the weights LEAVE the device (se_download / se_download_scaled on SE_SLOT_WOUT) —
  // round 1 ran a separate 8 B/row pass over WOUT for it (newton K1 0.76-0.87 of the HBM roofline because of that pass).
  const int dim = ctx->gbm.dim;
  std::vector<double> s((size_t)dim + 1);
  SE_TRY(gbm_fetch(ctx, 1 + dim, s.data()));
  ctx->wout_scale.assign((size_t)dim, 0.f);
  for (int j = 0; j < dim; ++j) {
    ctx->wout_scale[j] = (float)(1.0 / s[1 + j]);
    if (sum_hess) sum_hess[j] = s[1 + j];
  }
  ctx->wout_scaled = true;
  ctx->h_scal[0] = s[0];
  return SE_OK;
}

int se_gbm_pseudo_residuals(se_ctx* ctx, int newton, double* sum_hess) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  SE_REQUIRE(ctx, !newton || loss_has_hessian(ctx->gbm.loss), SE_ERR_ARG, "loss %d has no hessian (updates=newton)", ctx->gbm.loss);
  SE_TRY(begin(ctx));
  if (newton) SE_TRY(slot_alloc2d(ctx, SE_SLOT_WOUT, ctx->gbm.dim, ctx->gbm.n));
  GbmArgs a = gbm_args(ctx, false);
  ctx->wout_scaled = false;
  if (newton) a.ws = red_ws(ctx);  // Σ max(H,1e-2): reducing launch
  SE_TRY(gbm_launch(ctx, SE_KF_RESID, newton ? GBM_RESID_NEWTON : GBM_RESID, a, nullptr));
  if (newton) SE_TRY(newton_finish(ctx, sum_hess));
  ctx->gbm.r_current = true;  // squared loss: r = y - F for gradient and newton (h = 1) alike
  return end(ctx);
}

int se_gbm_linesearch_eval(se_ctx* ctx, const double* alpha, double* loss, double* grad) {
  if (!ctx || !alpha || !loss) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  const int dim = ctx->gbm.dim;
  GbmArgs a = gbm_args(ctx, false);
  if (ctx->ls_packed) {  // inside se_gbm_linesearch_brent: bit-identical 8 B/row view
    a.y = nullptr;
    a.F = ctx->d_ls_u;
    a.h = ctx->d_ls_v;
  }
  a.ws = red_ws(ctx);
  // Brent consumes the objective value only: skip the gradient/curvature arithmetic when nobody asked for it
  const int eval_mode = (!grad && ctx->gbm.loss != SE_LOSS_LOGLOSS) ? GBM_EVAL_LOSS : GBM_EVAL;
  SE_TRY(gbm_launch(ctx, SE_KF_EVAL, eval_mode, a, alpha));
  std::vector<double> s((size_t)dim + 1);
  SE_TRY(gbm_fetch(ctx, 1 + dim, s.data()));
  // lossSum is accumulated `dim` times per row in the reference (GBMLoss.scala:60-64)
  *loss = (double)dim * s[0] / ctx->gbm.wsum;
  if (grad)
    for (int j = 0; j < dim; ++j) grad[j] = s[1 + j] / ctx->gbm.wsum;
  return SE_OK;
}

int se_gbm_linesearch_stats(se_ctx* ctx, double* stats4) {
  if (!ctx || !stats4) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.loss == SE_LOSS_SQUARED, SE_ERR_STATE, "squared loss only");
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, false);
  a.stats_from_r = ctx->gbm.r_current ? 1 : 0;
  a.ws = red_ws(ctx);
  SE_LAUNCH_T(ctx, SE_KF_SQ_STATS, launch_gbm(SE_LOSS_SQUARED, GBM_SQ_STATS, a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  SE_TRY(fetch_scalars(ctx, 0, 3, stats4));
  stats4[3] = ctx->gbm.wsum;
  return SE_OK;
}

int se_gbm_update(se_ctx* ctx, const double* step, int flags, double* loss_sum, double* sum_hess) {
  if (!ctx || !step) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  const bool newton = (flags & SE_UPD_NEWTON) != 0;
  SE_REQUIRE(ctx, !newton || loss_has_hessian(ctx->gbm.loss), SE_ERR_ARG, "loss %d has no hessian", ctx->gbm.loss);
  SE_TRY(begin(ctx));
  if (newton) SE_TRY(slot_alloc2d(ctx, SE_SLOT_WOUT, ctx->gbm.dim, ctx->gbm.n));
  GbmArgs a = gbm_args(ctx, false);
  const int mode = newton ? GBM_UPDATE_NEWTON : ((flags & SE_UPD_RESIDUAL) ? GBM_UPDATE_RESID : GBM_UPDATE);
  if (newton) ctx->wout_scaled = false;
  a.ws = red_ws(ctx);
  SE_TRY(gbm_launch(ctx, SE_KF_UPDATE, mode, a, step));
  ctx->gbm.r_current = (mode != GBM_UPDATE);  // the fused modes refresh R from the new F
  if (newton) {
    SE_TRY(newton_finish(ctx, sum_hess));
    if (loss_sum) *loss_sum = ctx->h_scal[0];
    return end(ctx);
  }
  if ((flags & SE_UPD_LOSS) && loss_sum) return gbm_fetch(ctx, 1, loss_sum);
  return end(ctx);
}

int se_gbm_mean_loss(se_ctx* ctx, int which, double* out) {
  if (!ctx || !out) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  SE_REQUIRE(ctx, which == 0 || which == 1, SE_ERR_ARG, "which must be 0 (train) or 1 (validation)");
  SE_TRY(ensure_counts(ctx));
  // the GLOBAL count decides: a rank whose local shard is empty still launches the reduction (n = 0) so that the
  // collective of its peers completes
  SE_REQUIRE(ctx, (which == 1 ? ctx->gbm.nv_global : ctx->gbm.n_global) > 0.0, SE_ERR_ARG,
             which == 1 ? "no validation rows on any rank" : "no training rows on any rank");
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, which == 1);
  a.ws = red_ws(ctx);
  SE_TRY(gbm_launch(ctx, SE_KF_MEAN_LOSS, GBM_MEAN_LOSS, a, nullptr));
  double s = 0.0;
  SE_TRY(gbm_fetch(ctx, 1, &s));
  *out = s / (which == 1 ? ctx->gbm.nv_global : ctx->gbm.n_global);
  return SE_OK;
}

int se_gbm_update_validation(se_ctx* ctx, const double* step, double* mean_loss) {
  if (!ctx || !step) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on, SE_ERR_STATE, "se_gbm_configure first");
  SE_TRY(ensure_counts(ctx));
  SE_REQUIRE(ctx, ctx->gbm.nv_global > 0.0, SE_ERR_STATE, "no validation rows configured on any rank");
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, true);
  a.ws = red_ws(ctx);
  SE_TRY(gbm_launch(ctx, SE_KF_UPDATE, GBM_UPDATE, a, step));
  double s = 0.0;
  SE_TRY(gbm_fetch(ctx, 1, &s));
  if (mean_loss) *mean_loss = s / ctx->gbm.nv_global;
  return SE_OK;
}

namespace {
struct EvalClosure {
  se_ctx* ctx;
  int rc;
};
double eval_cb(double x, void* user) {
  EvalClosure* c = static_cast<EvalClosure*>(user);
  double l = NAN;
  if (c->rc == SE_OK) c->rc = se_gbm_linesearch_eval(c->ctx, &x, &l, nullptr);
  return l;
}
using Parabola = BrentParabola;
double parabola_cb(double x, void* user) { return (*static_cast<const Parabola*>(user))(x); }
}  // namespace

namespace {

int ensure_ls_view(se_ctx* ctx) {
  if (ctx->ls_cap >= ctx->gbm.n && ctx->d_ls_u) return SE_OK;
  if (ctx->d_ls_u) cudaFree(ctx->d_ls_u);
  ctx->d_ls_u = ctx->d_ls_v = nullptr;
  ctx->ls_cap = 0;
  // one allocation for both halves: a single L2 access-policy window covers the whole view
  const size_t half = ((size_t)ctx->gbm.n + 32 + 63) / 64 * 64;
  SE_CUDA(ctx, cudaMalloc(&ctx->d_ls_u, sizeof(float) * 2 * half));
  ctx->d_ls_v = ctx->d_ls_u + half;
  ctx->ls_cap = ctx->gbm.n;
  return SE_OK;
}

// One launch of the persistent line-search kernel (se_gbm_fused.cu): the whole Brent search (single == 0) or one
// evaluation of the objective at `start` with the tile direction of evaluation number `parity + 1` (single == 1).
int linesearch_persist(se_ctx* ctx, double lo, double hi, double start, double rel, double abs_tol, int max_eval,
                       int single, int parity, double* alpha, double* loss, int* n_eval) {
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  const int lossid = ctx->gbm.loss;
  const bool packed = gbm_linesearch_persist_packed(lossid);
  if (packed) SE_TRY(ensure_ls_view(ctx));
  LsArgs a;
  a.y = ctx->slot[SE_SLOT_Y].d;
  a.F = ctx->slot[SE_SLOT_F].d;
  a.h = ctx->slot[SE_SLOT_H].d;
  a.u = ctx->d_ls_u;
  a.v = ctx->d_ls_v;
  a.n = ctx->gbm.n;
  a.param = (float)ctx->gbm.param;
  a.wsum = ctx->gbm.wsum;
  a.lo = lo; a.hi = hi; a.start = start; a.rel = rel; a.abs_tol = abs_tol; a.max_eval = max_eval;
  a.single = single;
  a.timing = ctx->fused_timing;
  a.first_parity = parity;
  a.partials = ctx->d_partials;
  a.sync = ctx->d_fsync;
  a.epoch0 = ctx->fused_epoch;
  ctx->fused_epoch += (unsigned long long)(max_eval > 0 ? max_eval : 1) + 4;
  a.out = ctx->d_scal + kScalRound + 16;
  a.ws = red_ws(ctx, kScalRound + 16);  // takes ONE sequence number; the kernel uses seq, seq+1, ... per evaluation
  const unsigned long long seq0 = ctx->red_seq;
  LsLaunch cfg;
  // small shards (what strong scaling leaves per GPU) live entirely in shared memory + L2: fewer, fatter CTAs keep more
  // tiles resident and shorten the per-evaluation rendezvous (measured at 6.25 M rows: 0.355 ms/round with 3 CTAs/SM vs
  // 0.384 with 4; at 50 M rows 4 CTAs/SM are 12 % faster than 3)
  cfg.max_ctas_per_sm = (ctx->ls_ctas_per_sm == 4 && ctx->gbm.n <= 8000000) ? 3 : ctx->ls_ctas_per_sm;
  cfg.resident = ctx->ls_resident;
  cfg.ring = ctx->ls_ring;
  ctx->last_ls_hit_ratio = 0.0;
  if (packed && !single && ctx->l2_persist && ctx->l2_persist_max > 0 && ctx->l2_window_max > 0) {
    if (ctx->l2_persist_set != ctx->l2_persist_max) {
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, ctx->l2_persist_max) == cudaSuccess) ctx->l2_persist_set = ctx->l2_persist_max;
      cudaGetLastError();
    }
    if (ctx->l2_persist_set > 0) {
      size_t bytes = sizeof(float) * (size_t)(ctx->d_ls_v - ctx->d_ls_u) + sizeof(float) * (size_t)ctx->gbm.n;  // [u .. end of v)
      if (bytes > ctx->l2_window_max) bytes = ctx->l2_window_max;
      cfg.window_base = ctx->d_ls_u;
      cfg.window_bytes = bytes;
      const double want = ctx->l2_persist_frac * (double)ctx->l2_persist_set / (double)bytes;
      cfg.hit_ratio = (float)(want > 1.0 ? 1.0 : want);
      ctx->last_ls_hit_ratio = cfg.hit_ratio;
      ctx->l2_persist_dirty = true;
    }
  }
  int workers = 0;
  SE_LAUNCH_T(ctx, SE_KF_EVAL, launch_gbm_linesearch_persist(lossid, a, ctx->sms, cfg, ctx->stream, &workers));
  ctx->last_ls_workers = workers;
  double res[4] = {0, 0, 0, 0};
  const int rc = fetch_scalars(ctx, kScalRound + 16, 4, res);
  // every evaluation consumed one reduction sequence number on every rank (the first was taken by red_ws)
  const int passes = (int)res[3];
  if (ctx->p2p && ctx->nranks > 1 && passes > 1) ctx->red_seq = seq0 + (unsigned long long)(passes - 1);
  ctx->last_ls_passes = passes;
  if (ctx->fused_timing) {
    SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + kScalRound + 20, ctx->d_scal + kScalRound + 20, sizeof(double) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->last_fused_us[0] = ctx->h_scal[kScalRound + 20];  // worker passes
    ctx->last_fused_us[1] = ctx->h_scal[kScalRound + 21];  // fold + exchange + Brent step
    ctx->last_fused_us[2] = 0.0;
  }
  release_l2_persist(ctx);
  if (rc != SE_OK) return rc;
  if (alpha) *alpha = res[0];
  if (loss) *loss = res[1];
  if (n_eval) *n_eval = (int)fabs(res[2]);
  if (res[2] < 0.0) return fail(ctx, SE_ERR_OPT, "Brent exceeded MaxEval(%d)", max_eval);
  return SE_OK;
}

struct PersistEvalClosure {
  se_ctx* ctx;
  int rc;
  int k;  // evaluations so far
};
double persist_eval_cb(double x, void* user) {
  PersistEvalClosure* c = static_cast<PersistEvalClosure*>(user);
  double l = NAN;
  if (c->rc == SE_OK) c->rc = linesearch_persist(c->ctx, 0.0, 0.0, x, 1e-6, 1e-6, 1, /*single=*/1, /*parity=*/c->k, nullptr, &l, nullptr);
  c->k++;
  return l;
}

}  // namespace

int se_gbm_linesearch_brent(se_ctx* ctx, double lo, double hi, double start, double rel, double abs_tol,
                            int max_eval, double* alpha, double* loss, int* n_eval) {
  if (!ctx || !alpha) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.dim == 1, SE_ERR_STATE, "Brent line search needs dim == 1");
  if (ctx->gbm.loss == SE_LOSS_SQUARED) {
    double st[4];
    SE_TRY(se_gbm_linesearch_stats(ctx, st));
    Parabola p{st[0], st[1], st[2], st[3]};
    int rc = brent_impl(parabola_cb, &p, lo, hi, start, rel, abs_tol, max_eval, alpha, loss, n_eval);
    if (rc != SE_OK) return fail(ctx, rc, "Brent exceeded MaxEval(%d)", max_eval);
    return SE_OK;
  }
  // Default: ONE persistent launch runs all of Brent's evaluations on the device (no host round trip and no launch
  // per evaluation; tiles resident in shared memory / L2 between evaluations) — se_gbm_fused.cu.
  // (needs in-kernel cross-GPU sums: single GPU or the fused peer exchange, not the NCCL fallback)
  if (ctx->ls_mode != 0 && !ctx->gbm.use_bag && max_eval >= 1 && gbm_linesearch_persist_supported(ctx->gbm.loss) &&
      (ctx->nranks <= 1 || ctx->p2p)) {
    if (ctx->ls_mode == 1) return linesearch_persist(ctx, lo, hi, start, rel, abs_tol, max_eval, 0, 0, alpha, loss, n_eval);
    // mode 2: the HOST runs the same Brent template and asks the same kernel for one evaluation at a time; the
    // objective values, hence the iterates, must equal mode 1 bit for bit (tests/test_gpu_parity.py)
    PersistEvalClosure c{ctx, SE_OK, 0};
    int rc = brent_impl(persist_eval_cb, &c, lo, hi, start, rel, abs_tol, max_eval, alpha, loss, n_eval);
    if (c.rc != SE_OK) return c.rc;
    if (rc != SE_OK) return fail(ctx, rc, "Brent exceeded MaxEval(%d)", max_eval);
    return SE_OK;
  }
  // Round-1 path (one launch + one host poll per evaluation), kept for bags and as the A/B baseline.
  // Binary scalar losses depend on (2y-1)(F + αh) only: one 20 B/row pass builds u = (2y-1)F, v = (2y-1)h and
  // every one of Brent's 20-40 evaluations then reads 8 B/row instead of 12 — same values bit for bit
  // (multiplying by ±1 is exact and fma is sign-symmetric).
  const bool pack = (ctx->gbm.loss == SE_LOSS_BERNOULLI || ctx->gbm.loss == SE_LOSS_EXPONENTIAL) && max_eval >= 8 &&
                    !ctx->gbm.use_bag && getenv("SE_NO_LS_PACK") == nullptr;
  if (pack) {
    SE_CUDA(ctx, cudaSetDevice(ctx->device));
    SE_TRY(ensure_ls_view(ctx));
    SE_LAUNCH_T(ctx, SE_KF_OTHER, launch_gbm_pack_signed(ctx->slot[SE_SLOT_Y].d, ctx->slot[SE_SLOT_F].d, ctx->slot[SE_SLOT_H].d,
                                                         ctx->d_ls_u, ctx->d_ls_v, ctx->gbm.n, ctx->sms, ctx->stream));
    ctx->ls_packed = true;
  }
  EvalClosure c{ctx, SE_OK};
  int rc = brent_impl(eval_cb, &c, lo, hi, start, rel, abs_tol, max_eval, alpha, loss, n_eval);
  ctx->ls_packed = false;
  if (c.rc != SE_OK) return c.rc;
  if (rc != SE_OK) return fail(ctx, rc, "Brent exceeded MaxEval(%d)", max_eval);
  return SE_OK;
}

namespace {
// Squared loss: statistics kernel -> Brent on the device over the exact parabola (se_brent.cu, same template and
// rounding as the host line search) -> fused update reading alpha from device memory.  Three launches back to back,
// one host synchronisation per round (for alpha, the evaluation count and the train loss) instead of two.  Opt-in
// (SE_DEVICE_BRENT=1, see se_gbm_round).
int round_squared_device_brent(se_ctx* ctx, double learning_rate, double tol, int max_iter, int flags, double* alpha,
                               double* loss_sum, int* n_eval) {
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, false);
  a.stats_from_r = ctx->gbm.r_current ? 1 : 0;
  a.ws = red_ws(ctx, kScalRound);  // stats -> d_scal[kScalRound..+2], summed across GPUs
  SE_LAUNCH_T(ctx, SE_KF_SQ_STATS, launch_gbm(SE_LOSS_SQUARED, GBM_SQ_STATS, a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  SE_TRY(allreduce_dev(ctx, kScalRound, 3));
  double* out_dev = ctx->d_scal + kScalRound + 4;
  const bool mirror = ctx->use_mirror && ctx->h_mirror && (ctx->nranks <= 1 || ctx->p2p);
  constexpr int kMirrorBrent = 32;  // mirror slots [32..34]: above what any reducing kernel writes before its ticket
  SE_LAUNCH(ctx, launch_brent_parabola(ctx->d_scal + kScalRound, ctx->gbm.wsum, 0.0, 100.0, 1.0, tol, tol, max_iter,
                                       out_dev, mirror ? ctx->d_mirror + kMirrorBrent : nullptr, ctx->stream));
  GbmArgs u = gbm_args(ctx, false);
  u.dev_alpha = out_dev;
  u.lr64 = learning_rate;
  const int mode = (flags & SE_UPD_RESIDUAL) ? GBM_UPDATE_RESID : GBM_UPDATE;
  u.ws = red_ws(ctx);
  SE_LAUNCH_T(ctx, SE_KF_UPDATE, launch_gbm(SE_LOSS_SQUARED, mode, u, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  ctx->gbm.r_current = (mode != GBM_UPDATE);
  double ls = 0.0;
  SE_TRY(fetch_scalars(ctx, 0, 1, &ls));  // the line-search results were written before this kernel's ticket
  double res[3];
  if (mirror) {
    for (int i = 0; i < 3; ++i) res[i] = ctx->h_mirror[kMirrorBrent + i];
  } else {
    SE_CUDA(ctx, cudaMemcpyAsync(res, out_dev, sizeof(res), cudaMemcpyDeviceToHost, ctx->stream));
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if (res[2] < 0.0) return fail(ctx, SE_ERR_OPT, "Brent exceeded MaxEval(%d)", max_iter);
  if (alpha) *alpha = res[0];
  if (loss_sum) *loss_sum = ls;
  if (n_eval) *n_eval = (int)res[2];
  return SE_OK;
}
}  // namespace

namespace {
// Squared loss, one cooperative launch per round (se_gbm_fused.cu): statistics -> cross-GPU sum -> Brent -> update +
// residual + loss -> cross-GPU sum -> host mirror.  One launch and one host poll per round.
int round_squared_fused(se_ctx* ctx, double learning_rate, double tol, int max_iter, int flags, double* alpha,
                        double* loss_sum, int* n_eval) {
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  SqRoundArgs a;
  const auto& g = ctx->gbm;
  a.y = ctx->slot[SE_SLOT_Y].d;
  a.F = ctx->slot[SE_SLOT_F].d;
  a.h = ctx->slot[SE_SLOT_H].d;
  a.r = ctx->slot[SE_SLOT_R].d;
  a.bag = g.use_bag ? ctx->slot[SE_SLOT_BAG].d : nullptr;
  a.n = g.n;
  a.stats_from_r = g.r_current ? 1 : 0;
  a.l2_hints = ctx->l2_hints >= 0 ? ctx->l2_hints : (g.n <= kL2HintRows ? 1 : 0);
  a.lr = learning_rate;
  a.wsum = g.wsum;
  a.lo = 0.0; a.hi = 100.0; a.start = 1.0; a.rel = tol; a.abs_tol = tol; a.max_eval = max_iter;
  a.out = ctx->d_scal + kScalRound;
  // The train loss after the update follows from the (global) statistics in closed form — no second reduction, no
  // second cross-GPU exchange, and the host is served before the update phase ends.  With a bag the statistics run
  // over the bag while the loss runs over all rows: then the loss is reduced over the rows as in the two-launch path.
  const bool loss_reduce = g.use_bag || ctx->fused_loss_reduce;
  a.ws_a = red_ws(ctx, kScalRound);            // sequence number s (statistics)
  a.ws_a.host_out = nullptr;                   // the mirror ticket is written after Brent / the second reduction
  a.ws_a.host_flag = nullptr;
  if (ctx->mirror_valid) --ctx->mirror_ticket; // red_ws armed the mirror for ws_a: re-armed below
  constexpr int kMirrorRound = 32;             // mirror slots [32..38]: above what a reducing kernel writes before its ticket
  bool mirror = false;
  if (loss_reduce) {
    a.ws_b = red_ws(ctx, kScalRound + 8);      // sequence number s + 1 (loss), host mirror + ticket
    a.ws_b.partials = ctx->d_partials + (size_t)(kMaxGridPartials / 2) * 4;
    a.ws_b.counter = &ctx->d_fsync->counter_b;
    mirror = ctx->mirror_valid;
  } else {
    const bool global = ctx->last_reduce_global;  // keep what red_ws decided for the statistics
    mirror = ctx->use_mirror && ctx->h_mirror && (ctx->nranks <= 1 || ctx->p2p);
    if (mirror) {
      a.host_final = ctx->d_mirror;
      a.host_flag = reinterpret_cast<volatile unsigned long long*>(ctx->d_mirror + kMboxPayload);
      a.host_ticket = ++ctx->mirror_ticket;
      ctx->mirror_valid = true;
      ctx->mirror_off = kScalRound + 8;
    }
    ctx->last_reduce_global = global;
  }
  a.host_res = mirror ? ctx->d_mirror + kMirrorRound : nullptr;
  a.sync = ctx->d_fsync;
  a.epoch = ++ctx->fused_epoch;
  {
    // tiles of 16 KB per array; y and F are prefetched: 32 KB per tile, over at most fused_ctas_per_sm * sms CTAs
    const double per_cta = ctx->fused_prefetch_mb * 1e6 / (32768.0 * (double)(ctx->fused_ctas_per_sm * ctx->sms));
    a.prefetch_tiles = per_cta < 0.0 ? 0 : (per_cta > 64.0 ? 64 : (int)(per_cta + 0.5));
  }
  a.timing = ctx->fused_timing;
  a.l2_mode = ctx->fused_l2_mode == 1 ? 1 : 0;
  const int write_r = (flags & SE_UPD_RESIDUAL) ? 1 : 0;
  int grid = 0;
  void* wbase = nullptr;
  size_t wbytes = 0;
  if (ctx->fused_l2_mode == 2 && ctx->l2_persist_max > 0 && ctx->l2_window_max > 0) {
    wbytes = sizeof(float) * (size_t)g.n;
    if (wbytes > ctx->l2_window_max) wbytes = ctx->l2_window_max;
    if (wbytes > ctx->l2_persist_max) wbytes = ctx->l2_persist_max;
    if (ctx->l2_persist_set != wbytes) {
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, wbytes) == cudaSuccess) ctx->l2_persist_set = wbytes;
      cudaGetLastError();
    }
    wbase = a.r;
    ctx->l2_persist_dirty = true;
  }
  SE_LAUNCH_T(ctx, SE_KF_UPDATE, launch_gbm_round_sq_fused(a, write_r, loss_reduce ? 1 : 0, ctx->sms, ctx->fused_ctas_per_sm, ctx->stream,
                                                           &grid, wbase, wbytes));
  ctx->last_fused_grid = grid;
  ctx->gbm.r_current = write_r != 0;
  double ls = 0.0;
  SE_TRY(fetch_scalars(ctx, kScalRound + 8, 1, &ls));
  double res[7];
  if (mirror) {
    for (int i = 0; i < 7; ++i) res[i] = ctx->h_mirror[kMirrorRound + i];
  } else {
    SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + kScalRound, ctx->d_scal + kScalRound, sizeof(double) * 7, cudaMemcpyDeviceToHost, ctx->stream));
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 7; ++i) res[i] = ctx->h_scal[kScalRound + i];
  }
  for (int i = 0; i < 3; ++i) ctx->last_round_stats[i] = res[i];
  if (ctx->fused_timing) {
    double t[4];
    SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + kScalRound + 10, ctx->d_scal + kScalRound + 10, sizeof(double) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 4; ++i) t[i] = ctx->h_scal[kScalRound + 10 + i];
    ctx->last_fused_us[0] = t[1] - t[0]; ctx->last_fused_us[1] = t[2] - t[1]; ctx->last_fused_us[2] = t[3] - t[2];
  }
  if (alpha) *alpha = res[4];
  if (n_eval) *n_eval = (int)fabs(res[6]);
  if (loss_sum) *loss_sum = ls;
  if (res[6] < 0.0) return fail(ctx, SE_ERR_OPT, "Brent exceeded MaxEval(%d)", max_iter);
  return SE_OK;
}
}  // namespace

int se_gbm_round(se_ctx* ctx, double learning_rate, int optimized, double tol, int max_iter, int flags,
                 double* alpha, double* loss_sum, int* n_eval) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.dim == 1, SE_ERR_STATE, "se_gbm_round needs dim == 1");
  ctx->last_round_fused = 0;
  const bool sq_search = optimized && ctx->gbm.loss == SE_LOSS_SQUARED && !(flags & SE_UPD_NEWTON) && max_iter >= 1;
  if (sq_search) {
    // commons-math3 BrentOptimizer constructor checks (the host path performs them in brent_impl's caller)
    SE_REQUIRE(ctx, tol >= 2.0 * 2.220446049250313e-16 && tol > 0.0, SE_ERR_ARG, "tolerance %g too small for Brent", tol);
    // One cooperative launch per round (measured on B200: 52 vs 74 us at 12.5 M rows, 440 vs 454 us at 100 M rows).
    // With a communicator it needs the fused peer exchange (an NCCL all-reduce cannot run inside the kernel).
    const bool can = (ctx->nranks <= 1 || ctx->p2p);
    const bool want = ctx->fused_round > 0 || (ctx->fused_round < 0 && ctx->gbm.n <= ctx->fused_round_max_rows);
    if (can && want && getenv("SE_DEVICE_BRENT") == nullptr) {
      ctx->last_round_fused = 1;
      return round_squared_fused(ctx, learning_rate, tol, max_iter, flags, alpha, loss_sum, n_eval);
    }
  }
  // SE_DEVICE_BRENT=1: three launches (statistics, one-thread Brent, update) with one host synchronisation; kept as an
  // experiment switch — the fused round above supersedes it.
  if (sq_search && getenv("SE_DEVICE_BRENT") != nullptr)
    return round_squared_device_brent(ctx, learning_rate, tol, max_iter, flags, alpha, loss_sum, n_eval);
  double a = 1.0, obj = 0.0;
  int ne = 0;
  if (optimized) SE_TRY(se_gbm_linesearch_brent(ctx, 0.0, 100.0, 1.0, tol, tol, max_iter, &a, &obj, &ne));
  const double step = learning_rate * a;
  SE_TRY(se_gbm_update(ctx, &step, flags, loss_sum, nullptr));
  if (alpha) *alpha = a;
  if (n_eval) *n_eval = ne;
  return SE_OK;
}

int se_gbm_linesearch_eval2(se_ctx* ctx, double alpha, double* loss, double* d1, double* d2) {
  if (!ctx || !loss || !d1 || !d2) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.dim == 1 && ctx->gbm.loss != SE_LOSS_LOGLOSS, SE_ERR_STATE, "needs a dim-1 scalar loss");
  SE_TRY(ensure_wsum(ctx));
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, false);
  a.coef[0] = (float)alpha;
  a.ws = red_ws(ctx);
  SE_LAUNCH_T(ctx, SE_KF_EVAL, launch_gbm(ctx->gbm.loss, GBM_EVAL, a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  double s[3];
  SE_TRY(fetch_scalars(ctx, 0, 3, s));
  *loss = s[0] / ctx->gbm.wsum;
  *d1 = s[1] / ctx->gbm.wsum;
  *d2 = s[2] / ctx->gbm.wsum;
  return SE_OK;
}

int se_gbm_linesearch_newton(se_ctx* ctx, double lo, double hi, double start, double rel, double abs_tol,
                             int max_eval, double* alpha, double* loss, int* n_eval) {
  if (!ctx || !alpha) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.dim == 1, SE_ERR_STATE, "Newton line search needs dim == 1");
  SE_REQUIRE(ctx, loss_has_hessian(ctx->gbm.loss), SE_ERR_ARG, "loss %d has no hessian: use the Brent line search", ctx->gbm.loss);
  if (lo > hi) { const double t = lo; lo = hi; hi = t; }
  double a = lo, b = hi;
  double x = fmin(fmax(start, a), b);
  double f = NAN;
  int evals = 0;
  for (;;) {
    if (evals >= max_eval) return fail(ctx, SE_ERR_OPT, "Newton line search exceeded MaxEval(%d)", max_eval);
    double d1, d2;
    SE_TRY(se_gbm_linesearch_eval2(ctx, x, &f, &d1, &d2));
    ++evals;
    // the objective is convex along the line: the sign of the slope brackets the minimiser
    if (d1 > 0.0) b = x; else a = x;
    if ((x <= lo && d1 >= 0.0) || (x >= hi && d1 <= 0.0) || d1 == 0.0) break;  // boundary or stationary
    double xn = (d2 > 0.0) ? x - d1 / d2 : 0.5 * (a + b);
    // a Newton step that leaves the interval through an end that has not been evaluated yet: try that end
    // (a boundary minimum is then confirmed in one pass instead of ~20 bisections); otherwise bisect
    if (xn <= a) xn = (a == lo && x != lo) ? lo : 0.5 * (a + b);
    else if (xn >= b) xn = (b == hi && x != hi) ? hi : 0.5 * (a + b);
    if (fabs(xn - x) <= rel * fabs(x) + abs_tol) break;  // x is within tolerance of the minimiser
    x = xn;
  }
  *alpha = x;
  if (loss) *loss = f;
  if (n_eval) *n_eval = evals;
  return SE_OK;
}

int se_gbm_round_squared_async(se_ctx* ctx, double learning_rate) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->gbm.on && ctx->gbm.loss == SE_LOSS_SQUARED, SE_ERR_STATE, "squared loss only");
  SE_TRY(begin(ctx));
  GbmArgs a = gbm_args(ctx, false);
  a.stats_from_r = ctx->gbm.r_current ? 1 : 0;
  a.ws = red_ws(ctx, kScalRound);  // stats -> d_scal[kScalRound..+2]
  SE_LAUNCH_T(ctx, SE_KF_SQ_STATS, launch_gbm(SE_LOSS_SQUARED, GBM_SQ_STATS, a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  SE_TRY(allreduce_dev(ctx, kScalRound, 3));
  GbmArgs u = gbm_args(ctx, false);
  u.dev_stats = ctx->d_scal + kScalRound;
  u.lr = (float)learning_rate;
  u.ws = red_ws(ctx, kScalRound + 8);  // Σloss -> d_scal[kScalRound + 8]
  SE_LAUNCH_T(ctx, SE_KF_UPDATE, launch_gbm(SE_LOSS_SQUARED, GBM_UPDATE_RESID, u, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  SE_TRY(allreduce_dev(ctx, kScalRound + 8, 1));
  ctx->gbm.r_current = true;
  return end(ctx);
}

int se_gbm_round_result(se_ctx* ctx, double* alpha, double* loss_sum) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->h_scal + kScalRound, ctx->d_scal + kScalRound, sizeof(double) * 16,
                               cudaMemcpyDeviceToHost, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const double s1 = ctx->h_scal[kScalRound + 1], s2 = ctx->h_scal[kScalRound + 2];
  double al = (s2 > 0.0) ? s1 / s2 : 1.0;
  al = fmin(fmax(al, 0.0), 100.0);
  if (alpha) *alpha = al;
  if (loss_sum) *loss_sum = ctx->h_scal[kScalRound + 8];
  return SE_OK;
}

int se_brent_minimize(se_fn1 f, void* user, double lo, double hi, double start, double rel, double abs_tol,
                      int max_eval, double* x_out, double* f_out, int* n_eval) {
  if (!f) return fail(nullptr, SE_ERR_ARG, "null objective");
  // commons-math3 BrentOptimizer constructor checks
  if (rel < 2.0 * 2.220446049250313e-16) return fail(nullptr, SE_ERR_ARG, "relative threshold %g too small", rel);
  if (abs_tol <= 0.0) return fail(nullptr, SE_ERR_ARG, "absolute threshold must be > 0");
  int rc = brent_impl(f, user, lo, hi, start, rel, abs_tol, max_eval, x_out, f_out, n_eval);
  if (rc != SE_OK) return fail(nullptr, rc, "Brent exceeded MaxEval(%d)", max_eval);
  return SE_OK;
}

// ---- Spark's Bernoulli row sampler, restated (host only) -----------------------------------------
// RDD.sample(withReplacement = false, fraction, seed) as the reference calls it (regression/GBMRegressor.scala:357-359,
// classification/GBMClassifier.scala:329-331) for data that sits in ONE partition:
//   PartitionwiseSampledRDD: partition p gets the seed  new java.util.Random(seed).nextLong()  (p-th call);
//   BernoulliSampler.setSeed -> XORShiftRandom(seed'): state = hashSeed(seed') (MurmurHash3 of the 8 big-endian bytes);
//   sample(): fraction <= 0.4 -> GapSampling (skip floor(log(max(u, 5e-11)) / log1p(-fraction)) rows between picks),
//             else keep the row iff nextDouble() <= fraction.
// java.util.Random is specified by the Java SE API documentation; MurmurHash3 and XORShift are pinned by published
// vectors / their definitions (tests/test_thirdparty_golden.py); the sampler logic itself is restated from the Spark
// 3.3.1 sources (org/apache/spark/util/random/RandomSampler.scala, rdd/PartitionwiseSampledRDD.scala) and is UNPINNED
// (no Spark in this image).  A Spark host uploads the multiplicities Spark itself drew (GBMRegressorNative.scala).
namespace {
struct JavaRandom {
  uint64_t seed;
  explicit JavaRandom(int64_t s) : seed(((uint64_t)s ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1)) {}
  int32_t next(int bits) {
    seed = (seed * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
    return (int32_t)((int64_t)seed >> (48 - bits));
  }
  int64_t next_long() { const int64_t hi = next(32); const int64_t lo = next(32); return (int64_t)((uint64_t)hi << 32) + lo; }
};
uint32_t murmur3_bytes(const unsigned char* data, int len, uint32_t seed) {
  auto rotl = [](uint32_t x, int r) { return (x << r) | (x >> (32 - r)); };
  uint32_t h = seed;
  int i = 0;
  for (; len - i >= 4; i += 4) {
    uint32_t k = (uint32_t)data[i] | ((uint32_t)data[i + 1] << 8) | ((uint32_t)data[i + 2] << 16) | ((uint32_t)data[i + 3] << 24);
    k *= 0xcc9e2d51u; k = rotl(k, 15); k *= 0x1b873593u;
    h ^= k; h = rotl(h, 13); h = h * 5u + 0xe6546b64u;
  }
  uint32_t k = 0;
  const int rem = len - i;
  if (rem == 3) k ^= (uint32_t)data[i + 2] << 16;
  if (rem >= 2) k ^= (uint32_t)data[i + 1] << 8;
  if (rem >= 1) { k ^= (uint32_t)data[i]; k *= 0xcc9e2d51u; k = rotl(k, 15); k *= 0x1b873593u; h ^= k; }
  h ^= (uint32_t)len;
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
struct XorShift {
  uint64_t s;
  explicit XorShift(int64_t init) {
    unsigned char b[8];
    for (int i = 0; i < 8; ++i) b[i] = (unsigned char)((uint64_t)init >> (56 - 8 * i));  // ByteBuffer.putLong: big endian
    const uint32_t low = murmur3_bytes(b, 8, 0x3c074a61u);  // MurmurHash3.arraySeed
    const uint32_t high = murmur3_bytes(b, 8, low);
    s = ((uint64_t)high << 32) | (uint64_t)low;
  }
  int32_t next(int bits) {
    s ^= s << 21; s ^= s >> 35; s ^= s << 4;
    return (int32_t)(s & ((1ULL << bits) - 1));
  }
  double next_double() { return (double)(((int64_t)next(26) << 27) + next(27)) * (1.0 / (double)(1LL << 53)); }
};
}  // namespace

int se_spark_bernoulli_sample(int64_t seed, double fraction, int64_t n, int partition, float* counts) {
  if (!counts || n < 0 || partition < 0) return fail(nullptr, SE_ERR_ARG, "bad argument");
  JavaRandom jr(seed);
  int64_t pseed = 0;
  for (int p = 0; p <= partition; ++p) pseed = jr.next_long();
  XorShift rng(pseed);
  if (fraction <= 0.0) { for (int64_t i = 0; i < n; ++i) counts[i] = 0.f; return SE_OK; }
  if (fraction >= 1.0) { for (int64_t i = 0; i < n; ++i) counts[i] = 1.f; return SE_OK; }
  if (fraction <= 0.4) {  // RandomSampler.defaultMaxGapSamplingFraction
    const double lnq = log1p(-fraction), eps = 5e-11;  // RandomSampler.rngEpsilon
    auto advance = [&]() { const double u = fmax(rng.next_double(), eps); return (int64_t)(log(u) / lnq); };
    int64_t drop = advance();  // the GapSampling constructor advances once
    for (int64_t i = 0; i < n; ++i) {
      if (drop > 0) { --drop; counts[i] = 0.f; }
      else { drop = advance(); counts[i] = 1.f; }
    }
  } else {
    for (int64_t i = 0; i < n; ++i) counts[i] = (rng.next_double() <= fraction) ? 1.f : 0.f;
  }
  return SE_OK;
}

// ---- Boosting ----------------------------------------------------------------------------------
int se_boost_configure(se_ctx* ctx, int64_t n, int num_classes, int real) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, n >= 0 && num_classes >= 2, SE_ERR_ARG, "need n >= 0 and numClasses >= 2");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->boost.on = true; ctx->boost.n = n; ctx->boost.K = num_classes; ctx->boost.real = real != 0;
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_Y, 1, n));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_BW, 1, n));
  if (real) SE_TRY(slot_alloc2d(ctx, SE_SLOT_PROBA, num_classes, n));
  else SE_TRY(slot_alloc2d(ctx, SE_SLOT_PRED, 1, n));
  return SE_OK;
}

static BoostArgs boost_args(se_ctx* ctx, double sum_w) {
  release_l2_persist(ctx);
  ensure_labels_checked(ctx, 0, ctx->boost.K, ctx->boost.n);  // SAMME / SAMME.R compare (and index with) the label
  BoostArgs a;
  a.y = ctx->slot[SE_SLOT_Y].d;
  a.w = ctx->slot[SE_SLOT_BW].d;
  a.proba = ctx->slot[SE_SLOT_PROBA].d;
  a.pred = ctx->slot[SE_SLOT_PRED].d;
  a.n = ctx->boost.n;
  a.ld = ctx->slot[SE_SLOT_PROBA].ld;
  a.K = ctx->boost.K;
  a.inv_sum_w = (float)(1.0 / sum_w);
  a.ws = red_ws(ctx);
  return a;
}

int se_boost_real_update(se_ctx* ctx, double sum_w, double* est_err, double* new_sum) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->boost.on && ctx->boost.real, SE_ERR_STATE, "se_boost_configure(real=1) first");
  SE_TRY(begin(ctx));
  BoostArgs a = boost_args(ctx, sum_w);
  SE_LAUNCH_T(ctx, SE_KF_BOOST_REAL, launch_boost_real(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  double s[2];
  SE_TRY(fetch_scalars(ctx, 0, 2, s));
  if (est_err) *est_err = s[0];
  if (new_sum) *new_sum = s[1];
  return SE_OK;
}

int se_boost_discrete_error(se_ctx* ctx, double sum_w, double* est_err) {
  if (!ctx || !est_err) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->boost.on && !ctx->boost.real, SE_ERR_STATE, "se_boost_configure(real=0) first");
  SE_TRY(begin(ctx));
  BoostArgs a = boost_args(ctx, sum_w);
  SE_LAUNCH_T(ctx, SE_KF_BOOST_ERR, launch_boost_discrete_error(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  return fetch_scalars(ctx, 0, 1, est_err);
}

int se_boost_discrete_update(se_ctx* ctx, double sum_w, double beta, double* new_sum) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->boost.on && !ctx->boost.real, SE_ERR_STATE, "se_boost_configure(real=0) first");
  SE_TRY(begin(ctx));
  BoostArgs a = boost_args(ctx, sum_w);
  a.inv_beta = (float)(1.0 / beta);
  SE_LAUNCH_T(ctx, SE_KF_BOOST_UPD, launch_boost_discrete_update(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  double s = 0.0;
  SE_TRY(fetch_scalars(ctx, 0, 1, &s));
  if (new_sum) *new_sum = s;
  return SE_OK;
}

// ---- BoostingRegressor (AdaBoost.R2) -----------------------------------------------------------
int se_boostreg_configure(se_ctx* ctx, int64_t n) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, n >= 0, SE_ERR_ARG, "negative row count");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->boostreg.on = true;
  ctx->boostreg.n = n;
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_Y, 1, n));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_BW, 1, n));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_PRED, 1, n));
  return SE_OK;
}

static BoostRegArgs boostreg_args(se_ctx* ctx, double sum_w, int loss_type, double max_error, bool exchange = true) {
  release_l2_persist(ctx);
  BoostRegArgs a;
  a.y = ctx->slot[SE_SLOT_Y].d;
  a.pred = ctx->slot[SE_SLOT_PRED].d;
  a.w = ctx->slot[SE_SLOT_BW].d;
  a.n = ctx->boostreg.n;
  a.loss_type = loss_type;
  a.inv_sum_w = (float)(1.0 / sum_w);
  a.inv_max_err = (max_error == 0.0) ? 1.0f : (float)(1.0 / max_error);
  a.ws = red_ws(ctx, 0, exchange);
  return a;
}

int se_boostreg_max_error(se_ctx* ctx, double* max_error) {
  if (!ctx || !max_error) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->boostreg.on, SE_ERR_STATE, "se_boostreg_configure first");
  SE_TRY(begin(ctx));
  BoostRegArgs a = boostreg_args(ctx, 1.0, 0, 0.0, /*exchange=*/false);  // max-reduction: NCCL max afterwards
  SE_LAUNCH_T(ctx, SE_KF_OTHER, launch_boostreg_max(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  return fetch_scalars(ctx, 0, 1, max_error, kNcclMax);
}

int se_boostreg_error(se_ctx* ctx, double sum_w, int loss_type, double max_error, double* est_err) {
  if (!ctx || !est_err) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, ctx->boostreg.on, SE_ERR_STATE, "se_boostreg_configure first");
  SE_REQUIRE(ctx, loss_type >= SE_R2_EXPONENTIAL && loss_type <= SE_R2_SQUARED, SE_ERR_ARG, "bad loss type %d", loss_type);
  SE_TRY(begin(ctx));
  BoostRegArgs a = boostreg_args(ctx, sum_w, loss_type, max_error);
  SE_LAUNCH_T(ctx, SE_KF_BOOST_ERR, launch_boostreg_error(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  return fetch_scalars(ctx, 0, 1, est_err);
}

int se_boostreg_update(se_ctx* ctx, double sum_w, int loss_type, double max_error, double beta, double* new_sum) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->boostreg.on, SE_ERR_STATE, "se_boostreg_configure first");
  SE_REQUIRE(ctx, loss_type >= SE_R2_EXPONENTIAL && loss_type <= SE_R2_SQUARED, SE_ERR_ARG, "bad loss type %d", loss_type);
  SE_TRY(begin(ctx));
  BoostRegArgs a = boostreg_args(ctx, sum_w, loss_type, max_error);
  a.log2_beta = (float)log2(beta);
  SE_LAUNCH_T(ctx, SE_KF_BOOST_UPD, launch_boostreg_update(a, ctx->ctas_per_sm, ctx->sms, ctx->stream));
  double s = 0.0;
  SE_TRY(fetch_scalars(ctx, 0, 1, &s));
  if (new_sum) *new_sum = s;
  return SE_OK;
}

// ---- Aggregation -------------------------------------------------------------------------------
int se_agg_configure(se_ctx* ctx, int kind, int num_models, int num_classes, int dim, int loss, int64_t n) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, kind >= SE_AGG_GBM_REGRESSOR && kind <= SE_AGG_BOOSTING_REG_MEAN, SE_ERR_ARG, "bad kind %d", kind);
  SE_REQUIRE(ctx, num_models >= 0 && n >= 0, SE_ERR_ARG, "bad sizes");
  SE_CUDA(ctx, cudaSetDevice(ctx->device));
  auto& g = ctx->agg;
  g.on = true; g.kind = kind; g.M = num_models; g.K = num_classes; g.dim = dim; g.loss = loss; g.n = n;
  switch (kind) {
    case SE_AGG_GBM_REGRESSOR:
    case SE_AGG_BAGGING_REGRESSOR:
    case SE_AGG_BOOSTING_REG_MEAN: g.width = 1; g.C = 1; break;
    case SE_AGG_BOOSTING_REG_MEDIAN:
      SE_REQUIRE(ctx, num_models >= 1 && num_models <= 8192, SE_ERR_ARG, "weighted median supports 1..8192 models (got %d)", num_models);
      g.width = 1; g.C = 1; break;
    case SE_AGG_GBM_CLASSIFIER:
      SE_REQUIRE(ctx, dim >= 1 && num_classes >= 2, SE_ERR_ARG, "bad dim/numClasses");
      g.width = dim; g.C = (dim == 1 && num_classes == 2) ? 2 : dim; break;
    case SE_AGG_BAGGING_SOFT:
    case SE_AGG_BOOSTING_REAL:
      SE_REQUIRE(ctx, num_classes >= 2, SE_ERR_ARG, "numClasses >= 2");
      g.width = num_classes; g.C = num_classes; break;
    default:
      SE_REQUIRE(ctx, num_classes >= 2, SE_ERR_ARG, "numClasses >= 2");
      g.width = 1; g.C = num_classes; break;
  }
  const int64_t prow = (int64_t)(num_models > 0 ? num_models : 1) * g.width;
  // P is allocated with rows >= 2 semantics (padded stride) so every model row is 128 B aligned
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_P, prow, n));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_RAW, g.C, n));
  if (kind >= SE_AGG_GBM_CLASSIFIER && kind <= SE_AGG_BOOSTING_DISCRETE) {
    SE_TRY(slot_alloc2d(ctx, SE_SLOT_PROB, g.C, n));
    SE_TRY(slot_alloc2d(ctx, SE_SLOT_LABEL, 1, n));
  }
  return SE_OK;
}

int se_agg_run(se_ctx* ctx, const double* weights, const double* init) {
  if (!ctx) return fail(nullptr, SE_ERR_ARG, "null context");
  SE_REQUIRE(ctx, ctx->agg.on, SE_ERR_STATE, "se_agg_configure first");
  const auto& g = ctx->agg;
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  AggArgs a;
  a.kind = g.kind; a.M = g.M; a.K = g.K; a.dim = g.dim; a.loss = g.loss; a.n = g.n;
  a.P = ctx->slot[SE_SLOT_P].d; a.ld = ctx->slot[SE_SLOT_P].rows > 1 ? ctx->slot[SE_SLOT_P].ld : ctx->slot[SE_SLOT_P].cols;
  a.raw = ctx->slot[SE_SLOT_RAW].d;
  a.ld_out = ctx->slot[SE_SLOT_RAW].rows > 1 ? ctx->slot[SE_SLOT_RAW].ld : ctx->slot[SE_SLOT_RAW].cols;
  a.prob = ctx->slot[SE_SLOT_PROB].d;
  a.label = ctx->slot[SE_SLOT_LABEL].d;
  a.bad_label = ctx->d_bad_label;
  // small operands: narrowed to fp32 and staged through pinned memory into d_small
  float* hs = reinterpret_cast<float*>(ctx->h_small);
  size_t used = 0;
  const bool uses_w = (g.kind == SE_AGG_GBM_REGRESSOR || g.kind == SE_AGG_GBM_CLASSIFIER || g.kind == SE_AGG_BOOSTING_DISCRETE ||
                       g.kind == SE_AGG_BOOSTING_REG_MEAN || g.kind == SE_AGG_BOOSTING_REG_MEDIAN);
  const int nw = g.M * ((g.kind == SE_AGG_GBM_CLASSIFIER) ? g.dim : 1);
  SE_REQUIRE(ctx, (size_t)(nw + kMaxDim) * sizeof(float) * 2 <= (size_t)kSmallBytes, SE_ERR_ARG, "too many models");
  // the previous run may still be reading d_small/h_small
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (uses_w) {
    SE_REQUIRE(ctx, weights || g.M == 0, SE_ERR_ARG, "weights required for this aggregation kind");
    double sw = 0.0;
    for (int i = 0; i < nw; ++i) { hs[i] = (float)weights[i]; sw += (double)hs[i]; }  // Σ of what the device sees
    a.weights = reinterpret_cast<const float*>(ctx->d_small);
    a.sum_weights = sw;
    used = (size_t)nw;
  }
  if ((g.kind == SE_AGG_GBM_REGRESSOR || g.kind == SE_AGG_GBM_CLASSIFIER) && init) {
    const size_t off = (used + 31) / 32 * 32;
    for (int j = 0; j < g.dim; ++j) hs[off + j] = (float)init[j];
    a.init = reinterpret_cast<const float*>(ctx->d_small) + off;
    used = off + g.dim;
  }
  if (g.kind == SE_AGG_BOOSTING_REG_MEDIAN) {
    // cumulative weights are compared in fp64 like the reference: ship the weights as doubles too
    const size_t off = (used + 63) / 64 * 64;  // floats; keeps the doubles 8-byte aligned
    double* hd = reinterpret_cast<double*>(hs + off);
    for (int i = 0; i < g.M; ++i) hd[i] = weights[i];
    a.weights64 = reinterpret_cast<const double*>(reinterpret_cast<const float*>(ctx->d_small) + off);
    used = off + 2 * (size_t)g.M;
    // fast path (launch_agg): every weight finite and >= 0; all equal -> no rounding margin needed
    ctx->last_wm_mode = 0;
    if (ctx->wm_fast && g.M >= 1 && g.M <= 64 && g.n > 0) {
      bool ok = true, equal = true;
      for (int i = 0; i < g.M; ++i) {
        ok = ok && (weights[i] >= 0.0) && (weights[i] <= 1.7976931348623157e308);
        equal = equal && (weights[i] == weights[0]);
      }
      if (ok) {
        a.wm_mode = equal ? 2 : 1;
        a.weights64_host = weights;
        if (a.wm_mode == 1) {
          int64_t cap = ctx->wm_list_cap > 0 ? ctx->wm_list_cap : g.n / 4;
          if (cap < 1024 && ctx->wm_list_cap == 0) cap = 1024;
          if (cap > 2147483000LL) cap = 2147483000LL;
          if (ctx->wm_alloc < (size_t)cap + 1) {
            if (ctx->d_wm) cudaFree(ctx->d_wm);
            ctx->d_wm = nullptr; ctx->wm_alloc = 0;
            if (cudaMalloc(&ctx->d_wm, sizeof(unsigned int) * ((size_t)cap + 1)) == cudaSuccess) ctx->wm_alloc = (size_t)cap + 1;
            else cudaGetLastError();
          }
          if (ctx->d_wm) {
            a.wm_count = ctx->d_wm;
            a.wm_list = reinterpret_cast<int32_t*>(ctx->d_wm + 1);
            a.wm_cap = (unsigned int)cap;
          } else {
            a.wm_mode = 0;  // no room for the list: exact kernel
          }
        }
        ctx->last_wm_mode = a.wm_mode;
      }
    }
  }
  if (used) SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_small, hs, used * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  SE_LAUNCH_T(ctx, SE_KF_AGG, launch_agg(a, 8, ctx->sms, ctx->stream));
  if (g.kind == SE_AGG_GBM_CLASSIFIER || g.kind == SE_AGG_BAGGING_SOFT || g.kind == SE_AGG_BOOSTING_REAL)
    ctx->launches++;  // separate finalize kernel (the vote kinds fuse their epilogue)
  return end(ctx);
}

// ---- on-device base models ---------------------------------------------------------------------
namespace {
// Walk the uint8 rank matrix instead of the fp32 features when every threshold of the tree fits the per-column edge
// lists (<= 255 per column; Spark's trees draw theirs from the <= maxBins - 1 candidates of findSplits, the same on
// every round).  Returns 1 when the binned kernel was launched, 0 when the caller must take the fp32 walk.
// Makes the rank matrix of slot X cover every threshold of the given nodes (col[i] < 0: leaf): allocates it on first
// use, inserts new thresholds into the per-column edge lists and re-ranks the columns that changed.  Returns 1 when the
// matrix is ready, 0 when it cannot be used (disabled, no memory, NaN threshold, a column with more than 255 edges).
int bins_prepare(se_ctx* ctx, int which, const SlotBuf& X, int n_nodes, const int32_t* col, const float* thr) {
  ctx->last_tree_rebinned_cols = 0;
  if (!ctx->tree_bins || X.rows > 65535 || X.cols == 0) return 0;
  BinState& B = ctx->bins[which];
  const int d = (int)X.rows;
  if (!B.d8 || B.d != d || B.n != X.cols) {
    free_bins(B);
    const int64_t ld8 = ((X.cols + 127) / 128) * 128;
    bool ok = cudaMalloc(&B.d8, (size_t)d * (size_t)ld8) == cudaSuccess && cudaMalloc(&B.d_edges, sizeof(float) * 256 * (size_t)d) == cudaSuccess &&
              cudaMalloc(&B.d_nedges, sizeof(int32_t) * (size_t)d) == cudaSuccess && cudaMalloc(&B.d_cols, sizeof(int32_t) * (size_t)d) == cudaSuccess;
    if (!ok) {  // e.g. no room for another d x n bytes: keep walking the fp32 matrix
      cudaGetLastError();
      free_bins(B);
      ctx->tree_bins = 0;
      return 0;
    }
    B.ld8 = ld8; B.n = X.cols; B.d = d;
    B.edges.assign((size_t)d, std::vector<float>());
    B.dirty.assign((size_t)d, 0);
    B.valid = true;
  }
  if (!B.valid) {  // the slot was rewritten: every column that has edges must be re-ranked
    for (int c = 0; c < d; ++c) B.dirty[c] = B.edges[c].empty() ? 0 : 1;
    B.valid = true;
  }
  for (int i = 0; i < n_nodes; ++i) {
    if (col[i] < 0) continue;
    if (!(thr[i] == thr[i])) return 0;  // NaN threshold: leave it to the fp32 walk
    std::vector<float>& E = B.edges[col[i]];
    auto it = std::lower_bound(E.begin(), E.end(), thr[i]);
    if (it != E.end() && *it == thr[i]) continue;
    if (E.size() >= 255) return 0;      // this column needs more ranks than a byte holds
    E.insert(it, thr[i]);
    B.dirty[col[i]] = 1;
  }
  std::vector<int32_t> cols;
  for (int c = 0; c < d; ++c)
    if (B.dirty[c]) cols.push_back(c);
  if (!cols.empty()) {
    std::vector<int32_t> ne((size_t)d);
    for (int c = 0; c < d; ++c) ne[c] = (int32_t)B.edges[c].size();
    for (int32_t c : cols)
      SE_CUDA(ctx, cudaMemcpyAsync(B.d_edges + (size_t)c * 256, B.edges[c].data(), sizeof(float) * B.edges[c].size(), cudaMemcpyHostToDevice, ctx->stream));
    SE_CUDA(ctx, cudaMemcpyAsync(B.d_nedges, ne.data(), sizeof(int32_t) * (size_t)d, cudaMemcpyHostToDevice, ctx->stream));
    SE_CUDA(ctx, cudaMemcpyAsync(B.d_cols, cols.data(), sizeof(int32_t) * cols.size(), cudaMemcpyHostToDevice, ctx->stream));
    SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the host vectors above go out of scope
    BinArgs b;
    b.X = X.d; b.X8 = B.d8; b.n = X.cols; b.ld = X.rows > 1 ? X.ld : X.cols; b.ld8 = B.ld8;
    b.cols = B.d_cols; b.edges = B.d_edges; b.n_edges = B.d_nedges;
    SE_LAUNCH_T(ctx, SE_KF_OTHER, launch_bin_columns(b, (int)cols.size(), ctx->sms, ctx->stream));
    for (int32_t c : cols) B.dirty[c] = 0;
    ctx->last_tree_rebinned_cols = (int)cols.size();
  }
  return 1;
}

int tree_predict_binned(se_ctx* ctx, int which, const SlotBuf& X, int n_nodes, const int32_t* col, const float* thr,
                        const int32_t* left, const int32_t* right, const TreeArgs& t) {
  ctx->last_tree_binned = 0;
  ctx->last_tree_mask = 0;
  if (n_nodes > 65535) return 0;
  {
    const int rc = bins_prepare(ctx, which, X, n_nodes, col, thr);
    if (rc <= 0) return rc;
  }
  BinState& B = ctx->bins[which];
  if (B.nodes_cap < (size_t)n_nodes) {
    if (B.d_nodes) cudaFree(B.d_nodes);
    B.d_nodes = nullptr; B.nodes_cap = 0;
    SE_CUDA(ctx, cudaMalloc(&B.d_nodes, sizeof(uint4) * (size_t)n_nodes));
    B.nodes_cap = (size_t)n_nodes;
  }
  std::vector<uint4> nodes((size_t)n_nodes);
  int n_internal = 0;
  for (int i = 0; i < n_nodes; ++i) {
    if (col[i] < 0) { nodes[i] = make_uint4(0u, 0u, 0x80000000u, 0u); continue; }
    ++n_internal;
    const std::vector<float>& E = B.edges[col[i]];
    const uint32_t j = (uint32_t)(std::lower_bound(E.begin(), E.end(), thr[i]) - E.begin());  // x <= t_j  <=>  rank(x) <= j
    const uint64_t off = (uint64_t)col[i] * (uint64_t)B.ld8;
    nodes[i] = make_uint4((uint32_t)off, (uint32_t)(off >> 32), j, (uint32_t)left[i] | ((uint32_t)right[i] << 16));
  }
  SE_CUDA(ctx, cudaMemcpyAsync(B.d_nodes, nodes.data(), sizeof(uint4) * (size_t)n_nodes, cudaMemcpyHostToDevice, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  SE_LAUNCH_T(ctx, SE_KF_TREE, launch_tree_predict_binned(t, B.d8, B.d_nodes, n_internal, ctx->tree_mask, ctx->sms, ctx->stream));
  ctx->last_tree_binned = 1;
  ctx->last_tree_mask = (ctx->tree_mask && n_internal <= 64 && n_nodes <= 256) ? 1 : 0;
  return 1;
}
}  // namespace

static int tree_predict_impl(se_ctx* ctx, int which, int n_nodes, const int32_t* feature, const float* threshold,
                             const int32_t* left, const int32_t* right, const float* value, int n_out,
                             const int32_t* subspace, int n_subspace, int out_slot, int out_row) {
  if (!ctx || !feature || !threshold || !left || !right || !value) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, n_out >= 1 && n_out <= 4096, SE_ERR_ARG, "bad leaf width %d", n_out);
  const size_t bytes = (size_t)n_nodes * (16 + 4 * (size_t)n_out);
  SE_REQUIRE(ctx, n_nodes >= 1 && bytes <= (size_t)kSmallBytes && (size_t)n_nodes * 20 <= 200 * 1024,
             SE_ERR_ARG, "tree of %d nodes x %d outputs not supported", n_nodes, n_out);
  SE_REQUIRE(ctx, out_slot >= 0 && out_slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad out slot");
  const SlotBuf& X = ctx->slot[which ? SE_SLOT_VX : SE_SLOT_X];
  const SlotBuf& O = ctx->slot[out_slot];
  SE_REQUIRE(ctx, X.d, SE_ERR_STATE, "feature matrix slot not allocated");
  SE_REQUIRE(ctx, O.d && O.cols == X.cols && out_row >= 0 && out_row + n_out <= O.rows, SE_ERR_STATE, "output slot shape mismatch");
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int32_t* hf = reinterpret_cast<int32_t*>(ctx->h_small);
  float* ht = reinterpret_cast<float*>(hf + n_nodes);
  int32_t* hl = reinterpret_cast<int32_t*>(ht + n_nodes);
  int32_t* hr = hl + n_nodes;
  float* hv = reinterpret_cast<float*>(hr + n_nodes);
  for (int i = 0; i < n_nodes; ++i) {
    int32_t f = feature[i];
    if (f >= 0) {
      if (subspace) {
        SE_REQUIRE(ctx, f < n_subspace, SE_ERR_ARG, "node %d: feature %d outside subspace of %d", i, f, n_subspace);
        f = subspace[f];
      }
      SE_REQUIRE(ctx, f >= 0 && f < X.rows, SE_ERR_ARG, "node %d: column %d outside X with %lld columns", i, f, (long long)X.rows);
      SE_REQUIRE(ctx, left[i] >= 0 && left[i] < n_nodes && right[i] >= 0 && right[i] < n_nodes, SE_ERR_ARG, "node %d: bad child", i);
    }
    hf[i] = f; ht[i] = threshold[i]; hl[i] = left[i]; hr[i] = right[i];
  }
  // The device walk follows child links until it meets a leaf: reject anything that is not a tree rooted at node 0
  // (a node reached twice means a cycle or a DAG: the kernel could spin forever on it)
  {
    std::vector<char> seen((size_t)n_nodes, 0);
    std::vector<int32_t> stack;
    stack.push_back(0);
    seen[0] = 1;
    while (!stack.empty()) {
      const int32_t i = stack.back();
      stack.pop_back();
      if (hf[i] < 0) continue;  // leaf
      for (const int32_t c : {hl[i], hr[i]}) {
        SE_REQUIRE(ctx, !seen[c], SE_ERR_ARG, "node %d is reached twice (child of node %d): not a tree", c, i);
        seen[c] = 1;
        stack.push_back(c);
      }
    }
  }
  memcpy(hv, value, sizeof(float) * (size_t)n_nodes * n_out);
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_small, ctx->h_small, bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (out_slot == SE_SLOT_F || out_slot == SE_SLOT_R || out_slot == SE_SLOT_Y) ctx->gbm.r_current = false;
  TreeArgs t;
  t.X = X.d; t.n = X.cols; t.ld = X.rows > 1 ? X.ld : X.cols; t.n_nodes = n_nodes;
  t.feature = reinterpret_cast<const int32_t*>(ctx->d_small);
  t.threshold = reinterpret_cast<const float*>(t.feature + n_nodes);
  t.left = reinterpret_cast<const int32_t*>(t.threshold + n_nodes);
  t.right = t.left + n_nodes;
  t.value = reinterpret_cast<const float*>(t.right + n_nodes);
  t.n_out = n_out;
  t.ld_out = O.rows > 1 ? O.ld : O.cols;
  t.out = O.d + (int64_t)out_row * t.ld_out;
  {
    const int rc = tree_predict_binned(ctx, which, X, n_nodes, hf, ht, hl, hr, t);
    if (rc < 0) return rc;
    if (rc == 1) return end(ctx);
  }
  SE_LAUNCH_T(ctx, SE_KF_TREE, launch_tree_predict(t, ctx->sms, ctx->stream));
  return end(ctx);
}

int se_tree_predict(se_ctx* ctx, int which, int n_nodes, const int32_t* feature, const float* threshold,
                    const int32_t* left, const int32_t* right, const float* value,
                    const int32_t* subspace, int n_subspace, int out_slot, int out_row) {
  return tree_predict_impl(ctx, which, n_nodes, feature, threshold, left, right, value, 1, subspace, n_subspace,
                           out_slot, out_row);
}

int se_tree_predict_multi(se_ctx* ctx, int which, int n_nodes, const int32_t* feature, const float* threshold,
                          const int32_t* left, const int32_t* right, const float* values, int n_out,
                          const int32_t* subspace, int n_subspace, int out_slot) {
  return tree_predict_impl(ctx, which, n_nodes, feature, threshold, left, right, values, n_out, subspace, n_subspace,
                           out_slot, 0);
}

// ---- tree ensembles in one pass over the rank matrix (se_forest_predict, se_forest_classify) ----------------------
namespace {
// Every member must be a tree rooted at its first node, with tree-local child indices and GLOBAL column indices of X
// (the device walk follows child links until it meets a leaf: a node reached twice could make it spin forever).
int forest_validate(se_ctx* ctx, const SlotBuf& X, int n_trees, const int32_t* offsets, const int32_t* feature,
                    const int32_t* left, const int32_t* right) {
  SE_REQUIRE(ctx, n_trees >= 1 && n_trees <= (1 << 20), SE_ERR_ARG, "bad tree count %d", n_trees);
  SE_REQUIRE(ctx, offsets[0] == 0, SE_ERR_ARG, "offsets[0] must be 0");
  const int64_t total = offsets[n_trees];
  SE_REQUIRE(ctx, total >= n_trees && total <= (1 << 26), SE_ERR_ARG, "bad node count %lld", (long long)total);
  std::vector<char> seen;
  std::vector<int32_t> stack;
  for (int t = 0; t < n_trees; ++t) {
    const int32_t b = offsets[t], nn = offsets[t + 1] - offsets[t];
    SE_REQUIRE(ctx, nn >= 1 && nn <= 65535, SE_ERR_ARG, "tree %d: %d nodes (1..65535 supported)", t, nn);
    for (int i = 0; i < nn; ++i) {
      if (feature[b + i] < 0) continue;
      SE_REQUIRE(ctx, feature[b + i] < X.rows, SE_ERR_ARG, "tree %d node %d: column %d outside X with %lld columns", t, i,
                 feature[b + i], (long long)X.rows);
      SE_REQUIRE(ctx, left[b + i] >= 0 && left[b + i] < nn && right[b + i] >= 0 && right[b + i] < nn, SE_ERR_ARG,
                 "tree %d node %d: bad child", t, i);
    }
    seen.assign((size_t)nn, 0);
    stack.clear();
    stack.push_back(0);
    seen[0] = 1;
    while (!stack.empty()) {
      const int32_t i = stack.back();
      stack.pop_back();
      if (feature[b + i] < 0) continue;
      for (const int32_t c : {left[b + i], right[b + i]}) {
        SE_REQUIRE(ctx, !seen[c], SE_ERR_ARG, "tree %d: node %d is reached twice: not a tree", t, c);
        seen[c] = 1;
        stack.push_back(c);
      }
    }
  }
  return SE_OK;
}

// The forest kernels compare ranks, not features: every threshold of the forest must have a rank in the uint8 matrix.
int forest_ranks(se_ctx* ctx, int which, const SlotBuf& X, int64_t total, const int32_t* feature, const float* threshold) {
  const int rc = bins_prepare(ctx, which, X, (int)total, feature, threshold);
  if (rc < 0) return rc;
  SE_REQUIRE(ctx, rc == 1, SE_ERR_STATE,
             "the forest kernel needs the uint8 rank matrix (tree_bins on, <= 255 distinct thresholds per column, no NaN "
             "threshold): evaluate the members with se_tree_predict + se_agg_run instead");
  return SE_OK;
}

size_t pad_to(size_t v, size_t to) { return (v + to - 1) / to * to; }

// Grows the chunk of trees order[p0..p1) (order == nullptr: identity) tree by tree while bytes(trees, columns, nodes),
// the kernel's shared memory, fits the budget; a member that does not fit the four-CTAs-per-SM budget alone gets two,
// then one CTA per SM.  On return `used` lists the chunk's global columns and local[] maps them to their position.
// Returns p1 (== p0: even one tree does not fit).  whole: a budget is taken only when ALL trees [p0, n_trees) fit it
// (p1 < n_trees on return: the forest does not fit one chunk).
int forest_chunk(const int32_t* order, int p0, int n_trees, const int32_t* offsets, const int32_t* feature,
                 std::vector<int32_t>& local, std::vector<int32_t>& used, size_t& nodes,
                 size_t (*bytes)(size_t T, size_t C, size_t Nn), bool whole = false) {
  int p1 = p0;
  for (const size_t budget : {(size_t)kForestSmemBudget, (size_t)(100 * 1024), (size_t)(216 * 1024)}) {
    for (int32_t c : used) local[c] = -1;
    used.clear();
    nodes = 0;
    for (p1 = p0; p1 < n_trees; ++p1) {
      const int t = order ? order[p1] : p1;
      const int32_t b = offsets[t], nn = offsets[t + 1] - offsets[t];
      std::vector<int32_t> added;
      for (int i = 0; i < nn; ++i) {
        const int32_t c = feature[b + i];
        if (c >= 0 && local[c] < 0) { local[c] = (int32_t)(used.size() + added.size()); added.push_back(c); }
      }
      const size_t T = (size_t)(p1 - p0 + 1), C = used.size() + added.size(), Nn = nodes + (size_t)nn;
      if (bytes(T, C, Nn) > budget || C > 65535) {
        for (int32_t c : added) local[c] = -1;
        break;
      }
      used.insert(used.end(), added.begin(), added.end());
      nodes = Nn;
    }
    if (whole ? p1 == n_trees : p1 > p0) break;
  }
  return p1;
}

// Packed nodes of one tree: x = local column | rank threshold << 16 | leaf << 31; y = left | right << 16 (tree-local)
// for an internal node, the leaf's ordinal among the tree's leaves (node order) for a leaf.  Returns the leaf count.
int forest_pack_tree(const BinState& B, const std::vector<int32_t>& local, int32_t b, int32_t nn, const int32_t* feature,
                     const float* threshold, const int32_t* left, const int32_t* right, uint2* out) {
  int leaves = 0;
  for (int i = 0; i < nn; ++i) {
    const int32_t c = feature[b + i];
    if (c < 0) { out[i] = make_uint2(0x80000000u, (uint32_t)leaves++); continue; }
    const std::vector<float>& E = B.edges[c];
    const uint32_t j = (uint32_t)(std::lower_bound(E.begin(), E.end(), threshold[b + i]) - E.begin());  // x <= t_j <=> rank <= j
    out[i] = make_uint2((uint32_t)local[c] | (j << 16), (uint32_t)left[b + i] | ((uint32_t)right[b + i] << 16));
  }
  return leaves;
}

// Copies a packed chunk into ctx->d_forest (grown on demand).
int forest_upload_blob(se_ctx* ctx, const std::vector<unsigned char>& blob) {
  if (ctx->forest_cap < blob.size()) {
    if (ctx->d_forest) cudaFree(ctx->d_forest);
    ctx->d_forest = nullptr; ctx->forest_cap = 0;
    SE_CUDA(ctx, cudaMalloc(&ctx->d_forest, blob.size()));
    ctx->forest_cap = blob.size();
  }
  // the previous chunk's kernel may still be reading d_forest
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_forest, blob.data(), blob.size(), cudaMemcpyHostToDevice, ctx->stream));
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // blob is pageable host memory reused by the next chunk
  return SE_OK;
}

size_t forest_predict_bytes(size_t T, size_t C, size_t Nn) {
  return pad_to(8 * T + 8 * C + 8 * Nn + pad_to(4 * (T + 1), 8) + pad_to(4 * Nn, 16), 16) + C * kForestTile;
}

// se_forest_classify's blob (ForestClassArgs) with at most T classes in a chunk, the ranks and the parked leaves
size_t forest_classify_bytes(size_t T, size_t C, size_t Nn) {
  return pad_to(8 * T + 8 * T + 8 * C + 8 * Nn + 4 * (T + 1) + 4 * T + 4 * (T + 1), 16) + pad_to(C * kForestTile, 16) +
         T * kForestTile * sizeof(uint16_t);
}
// se_forest_weighted_median's shared memory: se_forest_predict's blob and ranks, then the parked keys (uint32)
size_t forest_wmedian_bytes(size_t T, size_t C, size_t Nn) {
  return pad_to(forest_predict_bytes(T, C, Nn), 16) + T * kForestTile * sizeof(uint32_t);
}
}  // namespace

// Σ_t weights[t] · tree_t(x) + init for every row in one pass over the rank matrix per chunk of trees
// (GBMRegressionModel.predict, regression/GBMRegressor.scala:531-539; BaggingRegressionModel.predict,
// regression/BaggingRegressor.scala:221-228 with weights 1 / M).
int se_forest_predict(se_ctx* ctx, int which, int n_trees, const int32_t* offsets, const int32_t* feature,
                      const float* threshold, const int32_t* left, const int32_t* right, const float* value,
                      const double* weights, double init, int out_slot, int out_row) {
  if (!ctx || !offsets || !feature || !threshold || !left || !right || !value) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, out_slot >= 0 && out_slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad out slot");
  const SlotBuf& X = ctx->slot[which ? SE_SLOT_VX : SE_SLOT_X];
  const SlotBuf& O = ctx->slot[out_slot];
  SE_REQUIRE(ctx, X.d, SE_ERR_STATE, "feature matrix slot not allocated");
  SE_REQUIRE(ctx, O.d && O.cols == X.cols && out_row >= 0 && out_row < O.rows, SE_ERR_STATE, "output slot shape mismatch");
  SE_TRY(forest_validate(ctx, X, n_trees, offsets, feature, left, right));
  const int64_t total = offsets[n_trees];
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  SE_TRY(forest_ranks(ctx, which, X, total, feature, threshold));
  BinState& B = ctx->bins[which];
  if (out_slot == SE_SLOT_F || out_slot == SE_SLOT_R || out_slot == SE_SLOT_Y) ctx->gbm.r_current = false;
  ForestArgs a;
  a.X8 = B.d8; a.n = X.cols; a.ld8 = B.ld8;
  a.out = O.d + (int64_t)out_row * (O.rows > 1 ? O.ld : O.cols);
  a.init = init;
  std::vector<int32_t> local((size_t)X.rows, -1);  // global column -> local column of the current chunk
  std::vector<int32_t> used;
  std::vector<unsigned char> blob;
  int chunks = 0;
  int t0 = 0;
  while (t0 < n_trees) {
    size_t nodes = 0;
    const int t1 = forest_chunk(nullptr, t0, n_trees, offsets, feature, local, used, nodes, forest_predict_bytes);
    SE_REQUIRE(ctx, t1 > t0, SE_ERR_ARG, "tree %d alone (%d nodes) does not fit the forest kernel's shared memory", t0,
               offsets[t0 + 1] - offsets[t0]);
    const size_t T = (size_t)(t1 - t0), C = used.size(), Nn = nodes;
    a.T = (int)T; a.C = (int)C;
    a.off_coloff = (int)(8 * T);
    a.off_nodes = a.off_coloff + (int)(8 * C);
    a.off_treeoff = a.off_nodes + (int)(8 * Nn);
    a.off_values = a.off_treeoff + (int)pad_to(4 * (T + 1), 8);
    a.blob_bytes = (int)pad_to((size_t)a.off_values + 4 * Nn, 16);
    a.off_ranks = a.blob_bytes;
    blob.assign((size_t)a.blob_bytes, 0);
    double* bw = reinterpret_cast<double*>(blob.data());
    unsigned long long* bco = reinterpret_cast<unsigned long long*>(blob.data() + a.off_coloff);
    uint2* bn = reinterpret_cast<uint2*>(blob.data() + a.off_nodes);
    int32_t* bto = reinterpret_cast<int32_t*>(blob.data() + a.off_treeoff);
    float* bv = reinterpret_cast<float*>(blob.data() + a.off_values);
    for (size_t c = 0; c < C; ++c) bco[c] = (unsigned long long)used[c] * (unsigned long long)B.ld8;
    size_t at = 0;
    for (int t = t0; t < t1; ++t) {
      const int32_t b = offsets[t], nn = offsets[t + 1] - offsets[t];
      bw[t - t0] = weights ? weights[t] : 1.0;
      bto[t - t0] = (int32_t)at;
      forest_pack_tree(B, local, b, nn, feature, threshold, left, right, bn + at);
      for (int i = 0; i < nn; ++i) bv[at + i] = value[b + i];
      at += (size_t)nn;
    }
    bto[T] = (int32_t)at;
    SE_TRY(forest_upload_blob(ctx, blob));
    a.blob = ctx->d_forest;
    a.accumulate = chunks > 0 ? 1 : 0;
    SE_LAUNCH_T(ctx, SE_KF_TREE, launch_forest_predict(a, ctx->sms, ctx->stream));
    ++chunks;
    t0 = t1;
  }
  ctx->last_forest_chunks = chunks;
  ctx->last_tree_binned = 1;
  return end(ctx);
}

// predictRaw / raw2probability / raw2prediction of a classifier ensemble of trees in one pass over the rank matrix per
// chunk of trees: the stage-1 class sums se_agg_run forms from the members' outputs (GBMClassifier.scala:567-589,
// BaggingClassifier.scala:260-283, BoostingClassifier.scala:348-382) go straight to RAW, then the aggregation's own
// epilogue turns them into raw, probability and label.  No [M][K][n] member outputs exist at any point.
int se_forest_classify(se_ctx* ctx, int which, int kind, int num_classes, int dim, int loss, int n_trees,
                       const int32_t* offsets, const int32_t* feature, const float* threshold, const int32_t* left,
                       const int32_t* right, const float* leaf, int leaf_width, const double* weights, const double* init) {
  if (!ctx || !offsets || !feature || !threshold || !left || !right || !leaf) return fail(ctx, SE_ERR_ARG, "null argument");
  const int K = num_classes;
  SE_REQUIRE(ctx, kind >= SE_AGG_GBM_CLASSIFIER && kind <= SE_AGG_BOOSTING_DISCRETE, SE_ERR_ARG,
             "kind %d is not a classifier aggregation", kind);
  SE_REQUIRE(ctx, K >= 2, SE_ERR_ARG, "numClasses >= 2");
  const bool gbm = kind == SE_AGG_GBM_CLASSIFIER;
  const bool labels = kind == SE_AGG_BAGGING_HARD || kind == SE_AGG_BOOSTING_DISCRETE;
  const int mode = gbm ? kForestScalarLeaves : labels ? kForestLabelLeaves : kForestVectorLeaves;
  const int want_width = (mode == kForestVectorLeaves) ? K : 1;
  SE_REQUIRE(ctx, leaf_width == want_width, SE_ERR_ARG, "kind %d takes leaves of width %d (got %d)", kind, want_width, leaf_width);
  SE_REQUIRE(ctx, !gbm || (dim >= 1 && n_trees % dim == 0), SE_ERR_ARG, "GBM: %d trees are not rounds of dim %d", n_trees, dim);
  SE_REQUIRE(ctx, !labels || K <= 65536, SE_ERR_ARG, "label leaves: at most 65536 classes (got %d)", K);
  SE_REQUIRE(ctx, weights || !(gbm || kind == SE_AGG_BOOSTING_DISCRETE), SE_ERR_ARG, "weights required for this aggregation kind");
  const SlotBuf& X = ctx->slot[which ? SE_SLOT_VX : SE_SLOT_X];
  SE_REQUIRE(ctx, X.d, SE_ERR_STATE, "feature matrix slot not allocated");
  SE_TRY(forest_validate(ctx, X, n_trees, offsets, feature, left, right));
  const int64_t total = offsets[n_trees];
  // a label leaf is a class index: checked here once per leaf instead of once per row on the device
  if (labels)
    for (int64_t i = 0; i < total; ++i) {
      if (feature[i] >= 0) continue;
      const float v = leaf[i];
      SE_REQUIRE(ctx, v >= 0.f && v < (float)K && v == floorf(v), SE_ERR_ARG, "node %lld: leaf label %g is not a class in [0, %d)",
                 (long long)i, (double)v, K);
    }
  const int S = gbm ? dim : K;                           // classes with a stage-1 sum
  const int Cout = (gbm && dim == 1 && K == 2) ? 2 : S;  // rows of RAW / PROB (binary GBM: (-F, F))
  const int M = gbm ? n_trees / dim : n_trees;
  // leaf table: every tree's leaves in node order, one value (GBM, label) or K values (class probabilities) each;
  // SAMME.R sums log(max(p, eps)) (BoostingClassifier.scala:352-354): formed here once per leaf, in fp64
  std::vector<int32_t> lbase((size_t)n_trees);
  std::vector<float> lv;
  for (int t = 0; t < n_trees; ++t) {
    lbase[t] = (int32_t)lv.size();
    for (int32_t i = offsets[t]; i < offsets[t + 1]; ++i) {
      if (feature[i] >= 0) continue;
      for (int k = 0; k < want_width; ++k) {
        const double p = leaf[(size_t)i * want_width + k];
        lv.push_back(kind == SE_AGG_BOOSTING_REAL ? (float)log(fmax(p, 2.220446049250313e-16)) : (float)p);
      }
      SE_REQUIRE(ctx, lv.size() <= (size_t)INT32_MAX, SE_ERR_ARG, "leaf table of more than 2^31 values");
    }
  }
  // GBM: tree t is models(t / dim)(t % dim) and adds to class t % dim only — order the trees class-major (rounds in model
  // order inside a class), so a chunk covers a contiguous range of classes; the other kinds add to every class.
  std::vector<int32_t> order((size_t)n_trees);
  for (int p = 0; p < n_trees; ++p) order[p] = gbm ? (p % M) * dim + p / M : p;
  double sum_a = 0.0;
  if (kind == SE_AGG_BOOSTING_DISCRETE)
    for (int t = 0; t < n_trees; ++t) sum_a += weights[t];
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  SE_TRY(forest_ranks(ctx, which, X, total, feature, threshold));
  BinState& B = ctx->bins[which];
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_RAW, Cout, X.cols));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_PROB, Cout, X.cols));
  SE_TRY(slot_alloc2d(ctx, SE_SLOT_LABEL, 1, X.cols));
  const SlotBuf& R = ctx->slot[SE_SLOT_RAW];
  if (ctx->forest_leaves_cap < lv.size()) {
    if (ctx->d_forest_leaves) cudaFree(ctx->d_forest_leaves);
    ctx->d_forest_leaves = nullptr; ctx->forest_leaves_cap = 0;
    SE_CUDA(ctx, cudaMalloc(&ctx->d_forest_leaves, sizeof(float) * lv.size()));
    ctx->forest_leaves_cap = lv.size();
  }
  SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_forest_leaves, lv.data(), sizeof(float) * lv.size(), cudaMemcpyHostToDevice, ctx->stream));
  ForestClassArgs a;
  a.X8 = B.d8; a.n = X.cols; a.ld8 = B.ld8;
  a.mode = mode; a.K = K;
  a.leaves = ctx->d_forest_leaves;
  a.raw = R.d; a.ld_raw = Cout > 1 ? R.ld : R.cols;
  std::vector<int32_t> local((size_t)X.rows, -1);
  std::vector<int32_t> used;
  std::vector<unsigned char> blob;
  int chunks = 0, p0 = 0, prev_last = -1;
  while (p0 < n_trees) {
    size_t nodes = 0;
    const int p1 = forest_chunk(order.data(), p0, n_trees, offsets, feature, local, used, nodes, forest_classify_bytes);
    SE_REQUIRE(ctx, p1 > p0, SE_ERR_ARG, "tree %d alone (%d nodes) does not fit the forest kernel's shared memory", order[p0],
               offsets[order[p0] + 1] - offsets[order[p0]]);
    const size_t T = (size_t)(p1 - p0), C = used.size(), Nn = nodes;
    // classes this chunk writes, and which of them continue a sum an earlier chunk left in RAW
    a.c0 = gbm ? order[p0] % dim : 0;
    a.c1 = gbm ? order[p1 - 1] % dim + 1 : S;
    a.acc0 = a.c0;
    a.acc1 = gbm ? (a.c0 == prev_last ? a.c0 + 1 : a.c0) : (chunks > 0 ? S : 0);
    const size_t NC = gbm ? (size_t)(a.c1 - a.c0) : 0;
    a.T = (int)T; a.C = (int)C;
    a.off_init = (int)(8 * T);
    a.off_coloff = a.off_init + (int)(8 * NC);
    a.off_nodes = a.off_coloff + (int)(8 * C);
    a.off_treeoff = a.off_nodes + (int)(8 * Nn);
    a.off_lbase = a.off_treeoff + (int)(4 * (T + 1));
    a.off_cstart = a.off_lbase + (int)(4 * T);
    a.blob_bytes = (int)pad_to((size_t)a.off_cstart + 4 * (NC + 1), 16);
    a.off_ranks = a.blob_bytes;
    a.off_parked = a.off_ranks + (int)pad_to(C * kForestTile, 16);
    blob.assign((size_t)a.blob_bytes, 0);
    double* bw = reinterpret_cast<double*>(blob.data());
    double* binit = reinterpret_cast<double*>(blob.data() + a.off_init);
    unsigned long long* bco = reinterpret_cast<unsigned long long*>(blob.data() + a.off_coloff);
    uint2* bn = reinterpret_cast<uint2*>(blob.data() + a.off_nodes);
    int32_t* bto = reinterpret_cast<int32_t*>(blob.data() + a.off_treeoff);
    int32_t* blb = reinterpret_cast<int32_t*>(blob.data() + a.off_lbase);
    int32_t* bcs = reinterpret_cast<int32_t*>(blob.data() + a.off_cstart);
    for (size_t c = 0; c < C; ++c) bco[c] = (unsigned long long)used[c] * (unsigned long long)B.ld8;
    for (size_t j = 0; j < NC; ++j) binit[j] = init ? init[a.c0 + j] : 0.0;
    size_t at = 0;
    for (int p = p0; p < p1; ++p) {
      const int t = order[p];
      const int32_t b = offsets[t], nn = offsets[t + 1] - offsets[t];
      bw[p - p0] = weights ? weights[t] : 1.0;  // GBM: weights[t] = a(t / dim)(t % dim); SAMME: a_t
      bto[p - p0] = (int32_t)at;
      blb[p - p0] = lbase[t];
      forest_pack_tree(B, local, b, nn, feature, threshold, left, right, bn + at);
      at += (size_t)nn;
      if (gbm) bcs[t % dim - a.c0 + 1] = p - p0 + 1;  // trees of class c: [cstart[c - c0], cstart[c - c0 + 1])
    }
    bto[T] = (int32_t)at;
    SE_TRY(forest_upload_blob(ctx, blob));
    a.blob = ctx->d_forest;
    SE_LAUNCH_T(ctx, SE_KF_TREE, launch_forest_classify(a, ctx->sms, ctx->stream));
    ++chunks;
    prev_last = a.c1 - 1;
    p0 = p1;
  }
  SE_LAUNCH_T(ctx, SE_KF_AGG, launch_agg_finalize(kind, Cout, K, dim, loss, M, sum_a, X.cols, a.ld_raw, R.d,
                                                  ctx->slot[SE_SLOT_PROB].d, ctx->slot[SE_SLOT_LABEL].d, ctx->sms,
                                                  ctx->stream));
  ctx->last_forest_chunks = chunks;
  ctx->last_tree_binned = 1;
  return end(ctx);
}

// AdaBoost.R2's weighted median of tree members (BoostingRegressionModel.predict, regression/BoostingRegressor.scala:
// 333-337; ensemble/Utils.scala:26-40) in one pass over the rank matrix: the value se_agg_run selects from the members'
// outputs, with the same mode choice and the same per-row code, without the [M][n] member outputs.
int se_forest_weighted_median(se_ctx* ctx, int which, int n_trees, const int32_t* offsets, const int32_t* feature,
                              const float* threshold, const int32_t* left, const int32_t* right, const float* value,
                              const double* weights, int out_slot, int out_row) {
  if (!ctx || !offsets || !feature || !threshold || !left || !right || !value) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, weights, SE_ERR_ARG, "weights required for the weighted median");
  SE_REQUIRE(ctx, out_slot >= 0 && out_slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad out slot");
  const SlotBuf& X = ctx->slot[which ? SE_SLOT_VX : SE_SLOT_X];
  const SlotBuf& O = ctx->slot[out_slot];
  SE_REQUIRE(ctx, X.d, SE_ERR_STATE, "feature matrix slot not allocated");
  SE_REQUIRE(ctx, O.d && O.cols == X.cols && out_row >= 0 && out_row < O.rows, SE_ERR_STATE, "output slot shape mismatch");
  SE_TRY(forest_validate(ctx, X, n_trees, offsets, feature, left, right));
  SE_REQUIRE(ctx, n_trees <= 64, SE_ERR_STATE,
             "%d trees: the one-pass weighted median takes at most 64 (evaluate the members with se_tree_predict + se_agg_run)",
             n_trees);
  // the whole forest must fit ONE chunk: a row's median needs every member's leaf at once
  std::vector<int32_t> local((size_t)X.rows, -1);  // global column -> local column
  std::vector<int32_t> used;
  size_t nodes = 0;
  const int t1 = forest_chunk(nullptr, 0, n_trees, offsets, feature, local, used, nodes, forest_wmedian_bytes, true);
  SE_REQUIRE(ctx, t1 == n_trees, SE_ERR_STATE,
             "the forest (%d trees, %lld nodes) does not fit one chunk of the weighted-median kernel's shared memory "
             "(evaluate the members with se_tree_predict + se_agg_run)", n_trees, (long long)offsets[n_trees]);
  const int64_t total = offsets[n_trees];
  // mode as se_agg_run picks it: every weight finite and >= 0 -> fast path, all equal -> no rounding margin
  int mode = 0;
  if (ctx->wm_fast && X.cols > 0) {
    bool ok = true, equal = true;
    for (int i = 0; i < n_trees; ++i) {
      ok = ok && (weights[i] >= 0.0) && (weights[i] <= 1.7976931348623157e308);
      equal = equal && (weights[i] == weights[0]);
    }
    if (ok) mode = equal ? 2 : 1;
  }
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  SE_TRY(forest_ranks(ctx, which, X, total, feature, threshold));
  BinState& B = ctx->bins[which];
  if (mode == 1 && !ctx->d_wm) {  // the deferred-row count lives where se_agg_run keeps it (d_wm[0])
    if (cudaMalloc(&ctx->d_wm, sizeof(unsigned int)) == cudaSuccess) ctx->wm_alloc = 1;
    else { cudaGetLastError(); ctx->d_wm = nullptr; mode = 0; }
  }
  if (out_slot == SE_SLOT_F || out_slot == SE_SLOT_R || out_slot == SE_SLOT_Y) ctx->gbm.r_current = false;
  const size_t T = (size_t)n_trees, C = used.size(), Nn = nodes;
  ForestWmArgs a;
  a.X8 = B.d8; a.n = X.cols; a.ld8 = B.ld8;
  a.out = O.d + (int64_t)out_row * (O.rows > 1 ? O.ld : O.cols);
  a.T = (int)T; a.C = (int)C;
  a.off_coloff = (int)(8 * T);
  a.off_nodes = a.off_coloff + (int)(8 * C);
  a.off_treeoff = a.off_nodes + (int)(8 * Nn);
  a.off_values = a.off_treeoff + (int)pad_to(4 * (T + 1), 8);
  a.blob_bytes = (int)pad_to((size_t)a.off_values + 4 * Nn, 16);
  a.off_ranks = a.blob_bytes;
  a.off_parked = a.off_ranks + (int)pad_to(C * kForestTile, 16);
  std::vector<unsigned char> blob((size_t)a.blob_bytes, 0);
  double* bw = reinterpret_cast<double*>(blob.data());
  unsigned long long* bco = reinterpret_cast<unsigned long long*>(blob.data() + a.off_coloff);
  uint2* bn = reinterpret_cast<uint2*>(blob.data() + a.off_nodes);
  int32_t* bto = reinterpret_cast<int32_t*>(blob.data() + a.off_treeoff);
  float* bv = reinterpret_cast<float*>(blob.data() + a.off_values);
  for (size_t c = 0; c < C; ++c) bco[c] = (unsigned long long)used[c] * (unsigned long long)B.ld8;
  size_t at = 0;
  for (int t = 0; t < n_trees; ++t) {
    const int32_t b = offsets[t], nn = offsets[t + 1] - offsets[t];
    bw[t] = weights[t];  // fp64, as se_agg_run ships them for the median
    bto[t] = (int32_t)at;
    forest_pack_tree(B, local, b, nn, feature, threshold, left, right, bn + at);
    for (int i = 0; i < nn; ++i) bv[at + i] = value[b + i];
    at += (size_t)nn;
  }
  bto[T] = (int32_t)at;
  SE_TRY(forest_upload_blob(ctx, blob));
  a.blob = ctx->d_forest;
  a.wm_mode = mode;
  a.weights_host = weights;
  a.deferred = mode == 1 ? ctx->d_wm : nullptr;
  SE_LAUNCH_T(ctx, SE_KF_TREE, launch_forest_wmedian(a, ctx->sms, ctx->stream));
  ctx->last_wm_mode = mode;
  ctx->last_forest_chunks = 1;
  ctx->last_tree_binned = 1;
  return end(ctx);
}

int se_linear_predict(se_ctx* ctx, int which, int n_coef, const float* coef, float intercept,
                      const int32_t* subspace, int out_slot, int out_row) {
  if (!ctx || (!coef && n_coef > 0)) return fail(ctx, SE_ERR_ARG, "null argument");
  SE_REQUIRE(ctx, n_coef >= 0 && (size_t)n_coef * 8 <= (size_t)kSmallBytes, SE_ERR_ARG, "bad coefficient count");
  SE_REQUIRE(ctx, out_slot >= 0 && out_slot < SE_NUM_SLOTS, SE_ERR_ARG, "bad out slot");
  const SlotBuf& X = ctx->slot[which ? SE_SLOT_VX : SE_SLOT_X];
  const SlotBuf& O = ctx->slot[out_slot];
  SE_REQUIRE(ctx, X.d, SE_ERR_STATE, "feature matrix slot not allocated");
  SE_REQUIRE(ctx, O.d && out_row >= 0 && out_row < O.rows && O.cols == X.cols, SE_ERR_STATE, "output slot shape mismatch");
  SE_TRY(begin(ctx));
  release_l2_persist(ctx);
  SE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  float* hc = reinterpret_cast<float*>(ctx->h_small);
  int32_t* hcol = reinterpret_cast<int32_t*>(hc + n_coef);
  for (int j = 0; j < n_coef; ++j) {
    hc[j] = coef[j];
    const int32_t col = subspace ? subspace[j] : j;
    SE_REQUIRE(ctx, col >= 0 && col < X.rows, SE_ERR_ARG, "column %d outside X", col);
    hcol[j] = col;
  }
  if (n_coef > 0)
    SE_CUDA(ctx, cudaMemcpyAsync(ctx->d_small, ctx->h_small, (size_t)n_coef * 8, cudaMemcpyHostToDevice, ctx->stream));
  const float* dc = reinterpret_cast<const float*>(ctx->d_small);
  const int32_t* dcol = reinterpret_cast<const int32_t*>(dc + n_coef);
  SE_LAUNCH_T(ctx, SE_KF_LINEAR, launch_linear_predict(X.d, X.cols, X.rows > 1 ? X.ld : X.cols, n_coef, dc, dcol, intercept,
                                       O.d + (int64_t)out_row * (O.rows > 1 ? O.ld : O.cols), ctx->sms, ctx->stream));
  return end(ctx);
}

}  // extern "C"
