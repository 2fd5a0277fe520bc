// se_agg.cu — ensemble Model.predict / predictRaw aggregation kernels (sm_100a).
//
// Reference per-row bodies (one JVM call per row through a UDF, SURVEY.md §3.4):
//   regression/GBMRegressor.scala:531-539        init + Σ_m a_m·P[m]
//   regression/BaggingRegressor.scala:221-228    (Σ_m P[m]) / M
//   classification/GBMClassifier.scala:564-589   res_j = init_j + Σ_m a_mj·P[m][j]; binary dim 1 -> (-res,res)
//   classification/BaggingClassifier.scala:260-287   soft: Σ_m p_m ; hard: Σ_m onehot(ŷ_m) ; prob = raw/M
//   classification/BoostingClassifier.scala:342-382  real: Σ_m (K-1)(ℓ_mk − mean_k ℓ_mk) ; discrete: ±a_m votes;
//                                                    prob = softmax(raw/(K-1))
//
// All of them are one streaming pass over the stacked base-model outputs P (the only large operand:
// 4·M·width B/row) followed by a tiny per-row epilogue.  Stage 1 (sum / vote histogram) is the
// HBM-bound kernel; stage 2 (finalize) touches only C values per row.
#include <stdlib.h>

#include "se_kernels.h"
#include "se_loss.cuh"
#include "se_tma.cuh"
#include "se_sortnet.h"
#include "se_wmedian.cuh"
#include "../../include/se_abi.h"

namespace se {

namespace {

constexpr float kSparkEps = 2.220446049250313e-16f;
constexpr int MU = 8;  // models loaded per batch: 8 independent 16 B requests per thread

// out[c][i] = init_c + Σ_m a[m][c] · f(P[m][c][i]),  f = identity or log(max(·,ε))
// P row (m,c) lives at P + (cols ? cols[m] : m*width + c) * ld.
template <bool LOGP>
__global__ void __launch_bounds__(kBlock) agg_sum_kernel(const float* __restrict__ P, int64_t n,
                                                        int64_t ld, int M, int width,
                                                        const float* __restrict__ a,
                                                        const float* __restrict__ init,
                                                        const int32_t* __restrict__ cols,
                                                        float post_div, float* __restrict__ out,
                                                        int64_t ld_out) {
  const int64_t n4 = n >> 2;
  for (int64_t g = (int64_t)blockIdx.x * kBlock + threadIdx.x; g < n4;
       g += (int64_t)gridDim.x * kBlock) {
    for (int c = 0; c < width; ++c) {
      // every batch of MU models is summed in fp32 (two short chains) and folded into fp64 accumulators: the
      // rounding error stays at the magnitude of one batch instead of growing with M (M = 512 in config 5)
      // (up to two batches there is nothing to gain: plain fp32 carry)
      const bool wide = M > 2 * MU;
      double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
      float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int m0 = 0; m0 < M; m0 += MU) {
        float4 v[MU];
        float wv[MU];
#pragma unroll
        for (int u = 0; u < MU; ++u) {
          const int m = m0 + u;
          if (m < M) {
            const int64_t rowi = cols ? (int64_t)cols[m] : (int64_t)m * width + c;
            v[u] = ld_stream4(P + rowi * ld + 4 * g);
            wv[u] = a ? a[(int64_t)m * width + c] : 1.0f;
          }
        }
        float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
#pragma unroll
        for (int u = 0; u < MU; ++u) {
          if (m0 + u < M) {
            float4 x = v[u];
            if (LOGP) {
              x.x = log_fast(fmaxf(x.x, kSparkEps)); x.y = log_fast(fmaxf(x.y, kSparkEps));
              x.z = log_fast(fmaxf(x.z, kSparkEps)); x.w = log_fast(fmaxf(x.w, kSparkEps));
            }
            float4& s = (u & 1) ? s1 : s0;  // two accumulator sets: shorter dependency chains
            s.x = fmaf(wv[u], x.x, s.x); s.y = fmaf(wv[u], x.y, s.y);
            s.z = fmaf(wv[u], x.z, s.z); s.w = fmaf(wv[u], x.w, s.w);
          }
        }
        if (wide) {
          d0 += (double)(s0.x + s1.x); d1 += (double)(s0.y + s1.y);
          d2 += (double)(s0.z + s1.z); d3 += (double)(s0.w + s1.w);
        } else {
          carry.x += s0.x + s1.x; carry.y += s0.y + s1.y; carry.z += s0.z + s1.z; carry.w += s0.w + s1.w;
        }
      }
      if (!wide) { d0 = (double)carry.x; d1 = (double)carry.y; d2 = (double)carry.z; d3 = (double)carry.w; }
      const double b = init ? (double)init[c] : 0.0;
      d0 += b; d1 += b; d2 += b; d3 += b;
      if (post_div != 0.f) { const double pd = (double)post_div; d0 /= pd; d1 /= pd; d2 /= pd; d3 /= pd; }
      const float4 r = make_float4((float)d0, (float)d1, (float)d2, (float)d3);
      st_stream4(out + c * ld_out + 4 * g, r);
    }
  }
  // tail rows
  const int tail = (int)(n & 3);
  if (blockIdx.x == 0 && threadIdx.x < tail) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    for (int c = 0; c < width; ++c) {
      double sd = init ? (double)init[c] : 0.0;
      for (int m = 0; m < M; ++m) {
        const int64_t rowi = cols ? (int64_t)cols[m] : (int64_t)m * width + c;
        float x = P[rowi * ld + i];
        if (LOGP) x = log_fast(fmaxf(x, kSparkEps));
        sd += (double)((a ? a[(int64_t)m * width + c] : 1.0f) * x);
      }
      if (post_div != 0.f) sd /= (double)post_div;
      out[c * ld_out + i] = (float)sd;
    }
  }
}

// Per-row epilogue on the C per-class sums t_c (from shared memory or from the RAW slot): raw, prob, label.
struct FinArgs {
  int kind, C, K, dim, loss, M;
  double sum_a;  // Σ a_m (boosting discrete)
  int64_t n, ld;
  float* raw;
  float* prob;
  float* label;
  int* bad_label;  // raised when a vote is not a class index in [0, K)
  double inv_km1;  // 1 / (K - 1)
};

// raw value from the stage-1 sum.  Real: the mean is a shift common to all classes (soft-max invariant), so fp32 is
// enough once the mean itself was accumulated in fp64; discrete: K·A_k − Σa subtracts nearly equal numbers and is
// formed in fp64 before the single rounding to the fp32 output.
template <class T>
__device__ __forceinline__ float fin_raw(const FinArgs& f, T t, float mean_t) {
  switch (f.kind) {
    case SE_AGG_BOOSTING_REAL:  // (K-1)(L_k − mean L)   BoostingClassifier.scala:355-360
      return (float)(f.K - 1) * ((float)t - mean_t);
    case SE_AGG_BOOSTING_DISCRETE:  // +a on the vote, −a/(K-1) elsewhere   :371-376
      return (float)(((double)t * (double)f.K - f.sum_a) * f.inv_km1);  // one reciprocal instead of an fp64 division per class
    default: return (float)t;
  }
}

// get(c) returns the stage-1 sum of class c for this row.  Two sweeps over the classes: (1) raw values with an
// online max / Σexp / first-argmax, (2) write raw and probability.
template <class Get>
__device__ __forceinline__ void finalize_row(const FinArgs& f, int64_t i, Get get) {
  const int C = f.C;
  float mean_t = 0.f;
  if (f.kind == SE_AGG_BOOSTING_REAL) {
    double s = 0.0;
    for (int c = 0; c < C; ++c) s += (double)get(c);
    mean_t = (float)(s / (double)C);
  }
  const bool softmax = (f.kind == SE_AGG_BOOSTING_REAL || f.kind == SE_AGG_BOOSTING_DISCRETE ||
                        f.kind == SE_AGG_GBM_CLASSIFIER);
  // boosting: softmax(raw/(K-1)) (BoostingClassifier.scala:342-346); GBM logloss: softmax(raw) (GBMLoss.scala:258-261)
  const float sc = (f.kind == SE_AGG_GBM_CLASSIFIER) ? kLog2e : kLog2e / (float)(f.K - 1);
  float best = -INFINITY, ssum = 0.f;
  int am = 0;
  for (int c = 0; c < C; ++c) {
    const float r = fin_raw(f, get(c), mean_t);
    if (r > best) am = c;  // Vector.argmax: first maximum
    const float mn = fmaxf(best, r);
    if (softmax) ssum = fmaf(ssum, ex2_approx((best - mn) * sc), ex2_approx((r - mn) * sc));
    best = mn;
  }
  f.label[i] = (float)am;
  const float inv = softmax ? rcp_approx(ssum) : 1.0f / (float)f.M;  // bagging: prob = raw·(1/M) (BaggingClassifier.scala:285-287)
  for (int c = 0; c < C; ++c) {
    const float r = fin_raw(f, get(c), mean_t);
    f.prob[c * f.ld + i] = softmax ? ex2_approx((r - best) * sc) * inv : r * inv;
    f.raw[c * f.ld + i] = r;
  }
}

// Vote histogram: A_c = Σ_{m: vote_m == c} a_m (a_m = 1 when a == nullptr).  One row per thread, per-thread
// histogram in shared memory laid out [K][kBlock] (conflict-free); the epilogue (raw, probability, argmax)
// runs straight out of shared memory — no intermediate [K][n] round trip through HBM.
// ncu / SASS on the first form of this kernel (weighted votes, M = 64, K = 26): 3860 instructions per row — per vote a
// 64-bit multiply for the address, a bounds predicate, a branch around the update and a global load + conversion of the
// model weight; per class an fp64 DIVISION in the epilogue.  This form walks the vote column with a pointer increment,
// stages the weights in shared memory in the histogram's type, updates branch-free (an invalid vote lands in a spare
// bin K and raises the error flag) and multiplies by 1/(K-1).
template <typename HT>  // float: unweighted counts (exact); double: weighted votes (error independent of M)
__global__ void __launch_bounds__(kBlock) agg_votes_kernel(const float* __restrict__ votes, int64_t ld, int M,
                                                          const float* __restrict__ a, const FinArgs f) {
  extern __shared__ __align__(8) unsigned char hist_raw[];
  HT* hist = reinterpret_cast<HT*>(hist_raw);  // [K + 1][kBlock]: bin K swallows invalid votes
  const int K = f.K;
  HT* s_a = hist + (size_t)(K + 1) * kBlock;    // [M] model weights (1 for plain votes)
  for (int m = threadIdx.x; m < M; m += kBlock) s_a[m] = a ? (HT)a[m] : (HT)1;
  __syncthreads();
  bool bad_vote = false;
  for (int64_t i0 = (int64_t)blockIdx.x * kBlock; i0 < f.n; i0 += (int64_t)gridDim.x * kBlock) {
    const int64_t i = i0 + threadIdx.x;
    HT* col = hist + threadIdx.x;
    for (int c = 0; c <= K; ++c) col[c * kBlock] = (HT)0;
    if (i < f.n) {
      const float* p = votes + i;
      int m0 = 0;
      for (; m0 + MU <= M; m0 += MU) {  // full batches: MU independent loads in flight, no per-vote predicates
        float v[MU];
#pragma unroll
        for (int u = 0; u < MU; ++u) v[u] = ld_stream1(p + (int64_t)u * ld);
        p += (int64_t)MU * ld;
#pragma unroll
        for (int u = 0; u < MU; ++u) {
          const int c = __float2int_rz(v[u]);
          const bool ok = ((unsigned)c < (unsigned)K) && ((float)c == v[u]);  // a vote is a predicted class index
          bad_vote = bad_vote || !ok;
          col[(ok ? c : K) * kBlock] += s_a[m0 + u];
        }
      }
      for (; m0 < M; ++m0, p += ld) {
        const float x = ld_stream1(p);
        const int c = __float2int_rz(x);
        const bool ok = ((unsigned)c < (unsigned)K) && ((float)c == x);
        bad_vote = bad_vote || !ok;
        col[(ok ? c : K) * kBlock] += s_a[m0];
      }
      // epilogue out of the thread's own histogram column, which doubles as fp32 scratch (ncu on the generic
      // two-sweep finalize_row: ~55 instructions per class; this form: 8 for plain votes, ~25 with the soft-max)
      float best = -INFINITY;
      int am = 0;
      if (f.kind == SE_AGG_BAGGING_HARD) {
        const float inv = 1.0f / (float)f.M;  // prob = raw·(1/M)  (BaggingClassifier.scala:285-287)
        for (int c = 0; c < K; ++c) {
          const float r = (float)col[c * kBlock];
          if (r > best) best = r, am = c;  // Vector.argmax: first maximum
          f.raw[c * f.ld + i] = r;
          f.prob[c * f.ld + i] = r * inv;
        }
      } else {
        const float sc = kLog2e / (float)(f.K - 1);  // prob = softmax(raw/(K-1))  (BoostingClassifier.scala:342-346)
        for (int c = 0; c < K; ++c) {
          const float r = fin_raw(f, col[c * kBlock], 0.f);
          if (r > best) best = r, am = c;
          f.raw[c * f.ld + i] = r;
          *reinterpret_cast<float*>(col + c * kBlock) = r;
        }
        float ssum = 0.f;
        for (int c = 0; c < K; ++c) {
          float* sp = reinterpret_cast<float*>(col + c * kBlock);
          const float e = ex2_approx((*sp - best) * sc);
          ssum += e;
          *sp = e;
        }
        const float inv = rcp_approx(ssum);
        for (int c = 0; c < K; ++c) f.prob[c * f.ld + i] = *reinterpret_cast<const float*>(col + c * kBlock) * inv;
      }
      f.label[i] = (float)am;
    }
  }
  if (bad_vote && f.bad_label != nullptr) *reinterpret_cast<volatile int*>(f.bad_label) = 1;
}

// Unweighted (hard) votes, the packed form: ncu on the histogram kernel above (M = 64, K = 26, 10 M rows): 2660
// instructions per row — 41 per vote — at 60 % issue utilisation and 47 % of the DRAM peak: issue-bound, not
// memory-bound.  Here a thread owns FOUR consecutive rows (one 128-bit load per model), counts are 8-bit fields packed
// four to a 32-bit word (class c -> word c >> 2, byte c & 3: M <= 255 never overflows a field), the words live in the
// thread's own shared-memory column (conflict-free, 4x less shared memory than one float per class), and the four
// rows give four independent read-modify-write chains.  Exact: integer counts.
constexpr int kVR = 4;  // rows per thread
__global__ void __launch_bounds__(kBlock) agg_hard_votes_packed_kernel(const float* __restrict__ votes, int64_t ld, int M,
                                                                      const FinArgs f) {
  extern __shared__ __align__(8) unsigned char hist_raw[];
  uint32_t* hist = reinterpret_cast<uint32_t*>(hist_raw);  // [W][kVR][kBlock]
  const int K = f.K;
  const int W = (K + 3) >> 2;
  bool bad_vote = false;
  const int64_t ngroups = (f.n + kVR - 1) / kVR;
  const float inv = 1.0f / (float)f.M;  // prob = raw·(1/M)  (BaggingClassifier.scala:285-287)
  for (int64_t g0 = (int64_t)blockIdx.x * kBlock; g0 < ngroups; g0 += (int64_t)gridDim.x * kBlock) {
    const int64_t g = g0 + threadIdx.x;
    for (int w = 0; w < W * kVR; ++w) hist[w * kBlock + threadIdx.x] = 0u;
    if (g >= ngroups) continue;
    const int64_t i0 = g * kVR;
    const bool full = (i0 + kVR <= f.n);  // rows are padded to 32 floats: the 128-bit load itself is always in bounds
    for (int m0 = 0; m0 < M; m0 += MU) {
      float4 v[MU];
#pragma unroll
      for (int u = 0; u < MU; ++u)
        if (m0 + u < M) v[u] = ld_stream4(votes + (int64_t)(m0 + u) * ld + i0);
#pragma unroll
      for (int u = 0; u < MU; ++u) {
        if (m0 + u >= M) break;
#pragma unroll
        for (int e = 0; e < kVR; ++e) {
          const float x = f4at(v[u], e);
          const int c = __float2int_rz(x);
          const bool ok = ((unsigned)c < (unsigned)K) && ((float)c == x);
          bad_vote = bad_vote || (!ok && (full || i0 + e < f.n));
          if (ok) hist[((c >> 2) * kVR + e) * kBlock + threadIdx.x] += 1u << ((c & 3) << 3);
        }
      }
    }
    // epilogue: one 128-bit store per class and output array for the thread's four rows
    int best[kVR] = {-1, -1, -1, -1}, am[kVR] = {0, 0, 0, 0};
    for (int c = 0; c < K; ++c) {
      float4 r;
#pragma unroll
      for (int e = 0; e < kVR; ++e) {
        const int cnt = (int)((hist[((c >> 2) * kVR + e) * kBlock + threadIdx.x] >> ((c & 3) << 3)) & 0xFFu);
        if (cnt > best[e]) best[e] = cnt, am[e] = c;  // Vector.argmax: first maximum
        f4at(r, e) = (float)cnt;
      }
      if (full) {
        st_stream4(f.raw + c * f.ld + i0, r);
        st_stream4(f.prob + c * f.ld + i0, make_float4(r.x * inv, r.y * inv, r.z * inv, r.w * inv));
      } else {
#pragma unroll
        for (int e = 0; e < kVR; ++e)
          if (i0 + e < f.n) {
            f.raw[c * f.ld + i0 + e] = f4at(r, e);
            f.prob[c * f.ld + i0 + e] = f4at(r, e) * inv;
          }
      }
    }
    if (full) {
      st_stream4(f.label + i0, make_float4((float)am[0], (float)am[1], (float)am[2], (float)am[3]));
    } else {
#pragma unroll
      for (int e = 0; e < kVR; ++e)
        if (i0 + e < f.n) f.label[i0 + e] = (float)am[e];
    }
  }
  if (bad_vote && f.bad_label != nullptr) *reinterpret_cast<volatile int*>(f.bad_label) = 1;
}

// (A four-rows-per-thread fp64 form of the WEIGHTED vote histogram was measured too: [K][4][128] doubles leave two
// 128-thread CTAs per SM and ran 2.81 ms vs 1.56 ms for agg_votes_kernel<double> at M = 64, K = 26, 10 M rows — the
// fp64 read-modify-write chains need the resident warps more than they need wider loads.  Not kept.)

// ------------------------------------------------------------------ class-wide sums through TMA tiles
// For the classifiers every row needs all C class sums before its epilogue (argmax, soft-max).  The streaming path
// (agg_sum_kernel + agg_finalize_kernel) round-trips a [C][n] intermediate through HBM and, per ncu, is
// instruction-bound: 15.8 instructions per element in stage 1 and 55 per (row, class) in the epilogue.  Here a W-warp
// CTA owns 128 W rows; the stacked model outputs arrive as 2-D tensor-map TMA boxes of G models x C classes x 128 W
// rows; a thread owns four rows and keeps the C x 4 sums of the current batch of <= 8 models in REGISTERS (one 128-bit
// shared-memory read and 4 FMAs — plus 4 lg2 for SAMME.R — per class and model); each batch is folded into the
// tile's running totals [C][128 W] in shared memory (own columns only), and the epilogue runs out of shared memory
// with 128-bit stores: P is read once, nothing is re-read.  Latency is covered by the other resident CTAs (up to 8
// per SM), not by per-CTA double buffering.
// W warps per CTA: 32 W threads, tiles of 128 W rows
constexpr int kAggMaxStages = 4;

struct ClassTileArgs {
  int M, C;          // models, classes
  int G;             // models per TMA box
  int stages;
  int logp;          // f = log max(p, eps) (boosting real)
  const float* a;    // weights [M][C] (GBM classifier) or null
  const float* init; // [C] or null
};

// epilogue of four rows whose C stage-1 sums sit in T[c * kAR + j] (this thread's own columns)
template <int kAR>
__device__ __forceinline__ void finalize_tile4(const FinArgs& f, float* T, int64_t row0) {
  const int C = f.C;
  const bool all_in = row0 + 3 < f.n;
  auto store4 = [&](float* base, const float4& v) {
    if (all_in) {
      st_stream4(base + row0, v);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (row0 + j < f.n) base[row0 + j] = f4at(v, j);
    }
  };
  float4 mean = make_float4(0.f, 0.f, 0.f, 0.f);
  if (f.kind == SE_AGG_BOOSTING_REAL) {
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
    for (int c = 0; c < C; ++c) {
      const float4 t = *reinterpret_cast<const float4*>(T + c * kAR);
      m0 += (double)t.x, m1 += (double)t.y, m2 += (double)t.z, m3 += (double)t.w;
    }
    const double ic = 1.0 / (double)C;
    mean = make_float4((float)(m0 * ic), (float)(m1 * ic), (float)(m2 * ic), (float)(m3 * ic));
  }
  const bool softmax = (f.kind == SE_AGG_BOOSTING_REAL || f.kind == SE_AGG_GBM_CLASSIFIER);
  const float sc = (f.kind == SE_AGG_GBM_CLASSIFIER) ? kLog2e : kLog2e / (float)(f.K - 1);
  // pass 1: raw (kept in the tile, written to HBM), max and first argmax
  float4 best = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  float4 am = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c = 0; c < C; ++c) {
    const float4 t = *reinterpret_cast<const float4*>(T + c * kAR);
    float4 r;
    r.x = fin_raw(f, t.x, mean.x), r.y = fin_raw(f, t.y, mean.y), r.z = fin_raw(f, t.z, mean.z), r.w = fin_raw(f, t.w, mean.w);
    const float cf = (float)c;  // Vector.argmax: first maximum
    if (r.x > best.x) best.x = r.x, am.x = cf;
    if (r.y > best.y) best.y = r.y, am.y = cf;
    if (r.z > best.z) best.z = r.z, am.z = cf;
    if (r.w > best.w) best.w = r.w, am.w = cf;
    *reinterpret_cast<float4*>(T + c * kAR) = r;
    store4(f.raw + c * f.ld, r);
  }
  store4(f.label, am);
  if (softmax) {
    float4 ssum = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < C; ++c) {
      const float4 r = *reinterpret_cast<const float4*>(T + c * kAR);
      float4 e;
      e.x = ex2_approx((r.x - best.x) * sc), e.y = ex2_approx((r.y - best.y) * sc);
      e.z = ex2_approx((r.z - best.z) * sc), e.w = ex2_approx((r.w - best.w) * sc);
      ssum.x += e.x, ssum.y += e.y, ssum.z += e.z, ssum.w += e.w;
      *reinterpret_cast<float4*>(T + c * kAR) = e;
    }
    const float4 inv = make_float4(rcp_approx(ssum.x), rcp_approx(ssum.y), rcp_approx(ssum.z), rcp_approx(ssum.w));
    for (int c = 0; c < C; ++c) {
      const float4 e = *reinterpret_cast<const float4*>(T + c * kAR);
      store4(f.prob + c * f.ld, make_float4(e.x * inv.x, e.y * inv.y, e.z * inv.z, e.w * inv.w));
    }
  } else {
    const float inv = 1.0f / (float)f.M;  // bagging: prob = raw·(1/M) (BaggingClassifier.scala:285-287)
    for (int c = 0; c < C; ++c) {
      const float4 r = *reinterpret_cast<const float4*>(T + c * kAR);
      store4(f.prob + c * f.ld, make_float4(r.x * inv, r.y * inv, r.z * inv, r.w * inv));
    }
  }
}

// dynamic shared memory (128-byte aligned): [stages][G*C][kAR] floats, then the running totals [C][kAR]
template <int CMAX, int W>
__global__ void __launch_bounds__(32 * W) agg_class_tile_kernel(const ClassTileArgs ta, const FinArgs f,
                                                             const __grid_constant__ CUtensorMap mapP) {
  constexpr int kAT = 32 * W, kAR = 128 * W;
  extern __shared__ __align__(128) unsigned char smem_dyn[];
  float* ring = reinterpret_cast<float*>(smem_dyn + ((128u - (smem_u32(smem_dyn) & 127u)) & 127u));
  __shared__ __align__(8) uint64_t full[kAggMaxStages];
  const int C = ta.C, M = ta.M, S = ta.stages;
  const int box_rows = ta.G * C;
  const int stage_floats = box_rows * kAR;
  const int tid = threadIdx.x;
  float* total = ring + (size_t)S * stage_floats + 4 * tid;  // this thread's four columns
  if (tid == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  (void)kAT;
  const int64_t ntiles = (f.n + kAR - 1) / kAR;
  const int64_t my_tiles = (ntiles > blockIdx.x) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int steps = (M + ta.G - 1) / ta.G;            // boxes per tile
  const int64_t nbox = my_tiles * steps;              // boxes this CTA consumes, in order
  auto issue = [&](int64_t q, int stage) {            // one elected thread
    const int64_t tile = blockIdx.x + (q / steps) * gridDim.x;
    const int step = (int)(q % steps);
    mbar_expect_tx(&full[stage], (uint32_t)(stage_floats * sizeof(float)));
    tma_load_tile_at(ring + (size_t)stage * stage_floats, &mapP, (int)(tile * kAR), step * box_rows, &full[stage]);
  };
  if (tid == 0)
    for (int s = 0; s < S && s < nbox; ++s) issue(s, s);

  const float fold_scale = ta.logp ? kLn2 : 1.0f;  // logs are summed in the lg2 domain
  int stage = 0;
  uint32_t phase = 0;
  int64_t q = 0;
  for (int64_t ti = 0; ti < my_tiles; ++ti) {
    const int64_t row0 = (blockIdx.x + ti * gridDim.x) * kAR + 4 * tid;
    float4 acc[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    int in_batch = 0;
    bool first_fold = true;
    for (int step = 0; step < steps; ++step, ++q) {
      mbar_wait(&full[stage], phase);
      const float* box = ring + (size_t)stage * stage_floats + 4 * tid;
      const int m0 = step * ta.G;
      const int gcount = min(ta.G, M - m0);
      for (int g = 0; g < gcount; ++g) {
        const float* bg = box + g * C * kAR;
        const float* wg = ta.a ? ta.a + (int64_t)(m0 + g) * C : nullptr;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
          if (c < C) {
            float4 x = *reinterpret_cast<const float4*>(bg + c * kAR);
            if (ta.logp) {
              x.x = lg2_approx(fmaxf(x.x, kSparkEps)), x.y = lg2_approx(fmaxf(x.y, kSparkEps));
              x.z = lg2_approx(fmaxf(x.z, kSparkEps)), x.w = lg2_approx(fmaxf(x.w, kSparkEps));
            }
            const float wv = wg ? __ldg(wg + c) : 1.0f;
            acc[c].x = fmaf(wv, x.x, acc[c].x), acc[c].y = fmaf(wv, x.y, acc[c].y);
            acc[c].z = fmaf(wv, x.z, acc[c].z), acc[c].w = fmaf(wv, x.w, acc[c].w);
          }
        }
      }
      __syncthreads();  // every thread is done with the box: the stage can be refilled
      if (tid == 0 && q + S < nbox) issue(q + S, stage);
      if (++stage == S) stage = 0, phase ^= 1;
      in_batch += gcount;
      if (in_batch >= 8 || step == steps - 1) {
        // fold the batch into the running totals: the rounding error stays at the magnitude of one batch
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
          if (c < C) {
            float4 t;
            if (first_fold) {
              const float b = ta.init ? __ldg(ta.init + c) : 0.f;
              t = make_float4(b, b, b, b);
            } else {
              t = *reinterpret_cast<const float4*>(total + c * kAR);
            }
            t.x = fmaf(acc[c].x, fold_scale, t.x), t.y = fmaf(acc[c].y, fold_scale, t.y);
            t.z = fmaf(acc[c].z, fold_scale, t.z), t.w = fmaf(acc[c].w, fold_scale, t.w);
            *reinterpret_cast<float4*>(total + c * kAR) = t;
            acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        first_fold = false;
        in_batch = 0;
      }
    }
    if (row0 < f.n) finalize_tile4<kAR>(f, total, row0);
  }
}

// Stage 2 for the sum-based kinds: per-row epilogue on tmp[C][n] (in RAW) -> raw, prob, label.
__global__ void __launch_bounds__(kBlock) agg_finalize_kernel(const FinArgs f) {
  for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < f.n;
       i += (int64_t)gridDim.x * kBlock) {
    if (f.kind == SE_AGG_GBM_CLASSIFIER && f.dim == 1 && f.K == 2) {
      // GBMClassifier.scala:583-584 + GBMLoss.scala:284-289,311-316 (raw(0) = −F)
      const float res = f.raw[i];
      const float r0 = -res;
      // p1 = 1/(1+e^x), p0 = 1 - p1 with x = raw(0) (bernoulli) or -2 raw(0) (exponential); both
      // formed from t = e^-|x| so the small one keeps full relative precision
      const float x = (f.loss == SE_LOSS_EXPONENTIAL) ? -2.0f * r0 : r0;
      const float t = exp_neg_fast(-fabsf(x));
      const float inv = rcp_approx(1.0f + t);
      const float p1 = (x >= 0.f) ? t * inv : inv;
      const float p0 = (x >= 0.f) ? inv : t * inv;
      f.raw[i] = r0;
      f.raw[f.ld + i] = res;
      f.prob[i] = p0;
      f.prob[f.ld + i] = p1;
      f.label[i] = (res > r0) ? 1.0f : 0.0f;  // argmax, first maximum on ties
      continue;
    }
    finalize_row(f, i, [&](int c) { return f.raw[c * f.ld + i]; });
  }
}

// Weighted median over M model outputs per row (ensemble/Utils.scala:26-40 via
// regression/BoostingRegressor.scala:333-337): stable sort of (value, weight) by value, cumulative weights in sorted
// order, first element whose cumulative weight reaches half of the total.
// One thread per row.  The row's M values become 64-bit words (order-preserving key << 32 | model index: all words
// distinct, ties keep model order = stable sort) in the thread's own column of shared memory [Mp][T] (conflict-free),
// padded to a power of two Mp with +inf words, and are sorted by a bitonic network — uniform control flow for the
// whole warp, O(M log² M) compare-exchanges instead of the O(M²) threshold scan it replaces (which was 0.07 of the
// HBM roofline at M = 32 because per-lane pruning diverges).  Total and running sums are then accumulated in fp64 in
// sorted order, exactly like the reference.
template <int T>
__global__ void __launch_bounds__(T) agg_wmedian_kernel(const float* __restrict__ P, int64_t n, int64_t ld, int M,
                                                       int Mp, const double* __restrict__ a,
                                                       float* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char wm_raw[];
  double* s_a = reinterpret_cast<double*>(wm_raw);                        // [M]
  unsigned long long* col = reinterpret_cast<unsigned long long*>(s_a + M) + threadIdx.x;  // [Mp][T], own column
  for (int m = threadIdx.x; m < M; m += T) s_a[m] = a[m];
  __syncthreads();
  for (int64_t r0 = (int64_t)blockIdx.x * T; r0 < n; r0 += (int64_t)gridDim.x * T) {
    const int64_t row = r0 + threadIdx.x;
    const bool in = row < n;
    for (int m = 0; m < Mp; ++m) {
      unsigned long long w = ~0ull;  // padding sorts last
      if (m < M) {
        const float v = in ? ld_stream1(P + (int64_t)m * ld + row) : 0.f;
        w = ((unsigned long long)wm_key(v) << 32) | (unsigned long long)(unsigned)m;
      }
      col[(size_t)m * T] = w;
    }
    // bitonic sort, ascending (own column only: no synchronisation)
    for (int k = 2; k <= Mp; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int e = 0; e < Mp; ++e) {
          const int l = e ^ j;
          if (l > e) {
            const unsigned long long x = col[(size_t)e * T], y = col[(size_t)l * T];
            const bool up = ((e & k) == 0);
            if ((x > y) == up) {
              col[(size_t)e * T] = y;
              col[(size_t)l * T] = x;
            }
          }
        }
      }
    }
    double total = 0.0;
    for (int m = 0; m < M; ++m) total += s_a[(unsigned)col[(size_t)m * T]];
    const double half = 0.5 * total;
    double cum = 0.0;
    unsigned long long pick = col[(size_t)(M - 1) * T];
    for (int m = 0; m < M; ++m) {
      const unsigned long long w = col[(size_t)m * T];
      cum += s_a[(unsigned)w];
      if (cum >= half) {
        pick = w;
        break;
      }
    }
    if (in) out[row] = wm_unkey((uint32_t)(pick >> 32));
  }
}

// Any number of models (M <= 8192): ONE WARP per row.  The row's words live in the warp's slice of shared memory and
// are sorted by a warp-cooperative bitonic network (lane e handles the pairs (e, e^j), e^j > e, 32 at a time); lane 0
// then accumulates the weights in sorted order, sequentially in fp64 — the reference's order (ensemble/Utils.scala:
// 26-40), so the selected element is identical.  The reference has no bound on M (JVM arrays); this is the general
// path behind the register (M <= 64) and thread-per-row (M <= 256) kernels.
constexpr int kWmWarps = 2;
__global__ void __launch_bounds__(32 * kWmWarps) agg_wmedian_warp_kernel(const float* __restrict__ P, int64_t n, int64_t ld,
                                                                         int M, int Mp, const double* __restrict__ a,
                                                                         float* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char wm_raw[];
  double* s_a = reinterpret_cast<double*>(wm_raw);  // [M]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* words = reinterpret_cast<unsigned long long*>(s_a + M) + (size_t)warp * Mp;  // [Mp], this warp's
  for (int m = threadIdx.x; m < M; m += 32 * kWmWarps) s_a[m] = a[m];
  __syncthreads();
  for (int64_t row = (int64_t)blockIdx.x * kWmWarps + warp; row < n; row += (int64_t)gridDim.x * kWmWarps) {
    for (int m = lane; m < Mp; m += 32) {
      unsigned long long w = ~0ull;  // padding sorts last
      if (m < M) w = ((unsigned long long)wm_key(ld_stream1(P + (int64_t)m * ld + row)) << 32) | (unsigned long long)(unsigned)m;
      words[m] = w;
    }
    __syncwarp();
    for (int k = 2; k <= Mp; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int e = lane; e < Mp; e += 32) {
          const int l = e ^ j;
          if (l > e) {
            const unsigned long long x = words[e], y = words[l];
            const bool up = ((e & k) == 0);
            if ((x > y) == up) {
              words[e] = y;
              words[l] = x;
            }
          }
        }
        __syncwarp();
      }
    }
    if (lane == 0) {
      double total = 0.0;
      for (int m = 0; m < M; ++m) total += s_a[(unsigned)words[m]];
      const double half = 0.5 * total;
      double cum = 0.0;
      unsigned long long pick = words[M - 1];
      for (int m = 0; m < M; ++m) {
        const unsigned long long w = words[m];
        cum += s_a[(unsigned)w];
        if (cum >= half) {
          pick = w;
          break;
        }
      }
      out[row] = wm_unkey((uint32_t)(pick >> 32));
    }
    __syncwarp();
  }
}

// Same algorithm with the row's words in REGISTERS (Mp <= 64): the network is fully unrolled, so every
// compare-exchange is ~6 ALU instructions and no memory traffic — the shared-memory form above moves 32 B per
// compare-exchange and thread and is bound by shared-memory bandwidth (measured 8.0 ms for 25 M rows at M = 32).
template <int MP>
__global__ void __launch_bounds__(128) agg_wmedian_reg_kernel(const __grid_constant__ CUtensorMap mapP, int64_t n,
                                                              int M, const double* __restrict__ a,
                                                              float* __restrict__ out) {
  // the sort is ALU work with no loads in flight, so the next tile of [M][128] values is prefetched into the other
  // shared-memory stage by one 2-D TMA box while the current tile is sorted (ncu on the direct-load form: 20 % issue
  // utilisation, long-scoreboard bound)
  extern __shared__ __align__(128) unsigned char wm_raw[];
  float* stage0 = reinterpret_cast<float*>(wm_raw + ((128u - (smem_u32(wm_raw) & 127u)) & 127u));
  const int stage_floats = M * 128;
  double* s_a = reinterpret_cast<double*>(stage0 + 2 * stage_floats);  // [M]
  __shared__ __align__(8) uint64_t full[2];
  if (threadIdx.x == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int m = threadIdx.x; m < M; m += 128) s_a[m] = a[m];
  __syncthreads();
  const int64_t ntiles = (n + 127) / 128;
  auto issue = [&](int64_t tile, int st) {
    mbar_expect_tx(&full[st], (uint32_t)(stage_floats * sizeof(float)));
    tma_load_tile(stage0 + (size_t)st * stage_floats, &mapP, (int)(tile * 128), &full[st]);
  };
  if (threadIdx.x == 0 && blockIdx.x < ntiles) issue(blockIdx.x, 0);
  uint32_t it = 0;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int st = it & 1;
    if (threadIdx.x == 0 && tile + gridDim.x < ntiles) issue(tile + gridDim.x, st ^ 1);  // freed by the barrier below
    const int64_t row = tile * 128 + threadIdx.x;
    const bool in = row < n;
    mbar_wait(&full[st], (it >> 1) & 1);
    const float* src = stage0 + (size_t)st * stage_floats + threadIdx.x;
    unsigned long long w[MP];
#pragma unroll
    for (int m = 0; m < MP; ++m) {
      w[m] = ~0ull;  // padding sorts last
      if (m < M) w[m] = ((unsigned long long)wm_key(src[m * 128]) << 32) | (unsigned long long)(unsigned)m;
    }
    __syncthreads();  // the tile is in registers: its stage may be refilled
    const unsigned long long pick = wm_exact_pick<MP>(w, M, s_a);
    if (in) out[row] = wm_unkey((uint32_t)(pick >> 32));
  }
}

// ---- weighted median, fast path (M <= 64, all weights finite and >= 0): see se_wmedian.cuh ---------------------
template <int MP>
__global__ void __launch_bounds__(128) agg_wmedian_fast_kernel(const __grid_constant__ CUtensorMap mapP, int64_t n, int M,
                                                               const __grid_constant__ WmWeights wts, double total,
                                                               double tau, int32_t* __restrict__ list,
                                                               unsigned int* __restrict__ count, unsigned int cap,
                                                               float* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char wm_raw[];
  float* stage0 = reinterpret_cast<float*>(wm_raw + ((128u - (smem_u32(wm_raw) & 127u)) & 127u));
  const int stage_floats = M * 128;
  __shared__ __align__(8) uint64_t full[2];
  if (threadIdx.x == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int64_t ntiles = (n + 127) / 128;
  auto issue = [&](int64_t tile, int st) {
    mbar_expect_tx(&full[st], (uint32_t)(stage_floats * sizeof(float)));
    tma_load_tile(stage0 + (size_t)st * stage_floats, &mapP, (int)(tile * 128), &full[st]);
  };
  if (threadIdx.x == 0 && blockIdx.x < ntiles) issue(blockIdx.x, 0);
  const double half = 0.5 * total;
  constexpr int LOG = (MP == 1) ? 0 : (MP == 2) ? 1 : (MP == 4) ? 2 : (MP == 8) ? 3 : (MP == 16) ? 4 : (MP == 32) ? 5 : 6;
  uint32_t it = 0;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int st = it & 1;
    if (threadIdx.x == 0 && tile + gridDim.x < ntiles) issue(tile + gridDim.x, st ^ 1);  // freed by the barrier below
    const int64_t row = tile * 128 + threadIdx.x;
    const bool in = row < n;
    mbar_wait(&full[st], (it >> 1) & 1);
    const float* src = stage0 + (size_t)st * stage_floats + threadIdx.x;
    uint32_t key[MP], s[MP];
#pragma unroll
    for (int m = 0; m < MP; ++m) {
      key[m] = 0xFFFFFFFFu;  // padding sorts last and carries weight 0
      if (m < M) key[m] = wm_key(src[m * 128]);
      s[m] = key[m];
    }
    __syncthreads();  // the tile is in registers: its stage may be refilled
    sortnet_oddeven<MP>(s, [](uint32_t& x, uint32_t& y) {
      const uint32_t lo = min(x, y), hi = max(x, y);
      x = lo;
      y = hi;
    });
    // invariant: P(lo) false, P(hi) true with P(k) := Ĉ(s[k]) >= ĥ; lo = t - 1, hi = t after LOG probes
    uint32_t t = 0, v_hi = s[MP - 1];
    double c_lo = 0.0, c_hi = total;
    auto probe = [&](uint32_t v) {
      double c = 0.0;
#pragma unroll
      for (int m = 0; m < MP; ++m) {
        // model order; padding (and m >= M) weights are 0.  fma(w, 1.0 or 0.0, c) is c + w rounded once, or c: one
        // select of the high word of the 0/1 factor instead of the two selects `if (...) c += w` compiles to
        const double b = __hiloint2double((key[m] <= v) ? 0x3ff00000 : 0, 0);
        c = fma(wts.w[m], b, c);
      }
      const bool right = !(c >= half);
      c_lo = right ? c : c_lo;
      c_hi = right ? c_hi : c;
      v_hi = right ? v_hi : v;
      t = 2u * t + (right ? 1u : 0u);
    };
    if constexpr (LOG > 0) probe(wm_candidate<MP, 0>(s, t));
    if constexpr (LOG > 1) probe(wm_candidate<MP, 1>(s, t));
    if constexpr (LOG > 2) probe(wm_candidate<MP, 2>(s, t));
    if constexpr (LOG > 3) probe(wm_candidate<MP, 3>(s, t));
    if constexpr (LOG > 4) probe(wm_candidate<MP, 4>(s, t));
    if constexpr (LOG > 5) probe(wm_candidate<MP, 5>(s, t));
    const bool safe = (c_hi - half > tau) && (half - c_lo > tau);
    if (in) out[row] = wm_unkey(v_hi);
    // rows whose decision could depend on the order of summation go to the exact kernel (warp-aggregated append)
    const bool defer = in && list != nullptr && !safe;
    const unsigned mask = __ballot_sync(0xffffffffu, defer);
    if (mask) {
      const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
      unsigned base = 0;
      if (lane == leader) base = atomicAdd(count, (unsigned)__popc(mask));
      base = __shfl_sync(0xffffffffu, base, leader);
      const unsigned idx = base + (unsigned)__popc(mask & ((1u << lane) - 1u));
      if (defer && idx < cap) list[idx] = (int32_t)row;
    }
  }
}

// exact pass over the deferred rows (or over ALL rows when the list overflowed): gathers, (key, model) words, the
// reference's sorted-order sums
template <int MP>
__global__ void __launch_bounds__(128) agg_wmedian_list_kernel(const float* __restrict__ P, int64_t n, int64_t ld, int M,
                                                               const double* __restrict__ a,
                                                               const int32_t* __restrict__ list,
                                                               const unsigned int* __restrict__ count, unsigned int cap,
                                                               float* __restrict__ out) {
  __shared__ double s_a[64];
  for (int m = threadIdx.x; m < 64; m += 128) s_a[m] = (m < M) ? a[m] : 0.0;
  __syncthreads();
  const unsigned int c = *count;
  if (c == 0) return;
  const bool all = c > cap;
  const int64_t items = all ? n : (int64_t)c;
  for (int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x; i < items; i += (int64_t)gridDim.x * 128) {
    const int64_t row = all ? i : (int64_t)list[i];
    unsigned long long w[MP];
#pragma unroll
    for (int m = 0; m < MP; ++m) {
      w[m] = ~0ull;
      if (m < M) w[m] = ((unsigned long long)wm_key(__ldg(P + (int64_t)m * ld + row)) << 32) | (unsigned long long)(unsigned)m;
    }
    out[row] = wm_unkey((uint32_t)(wm_exact_pick<MP>(w, M, s_a) >> 32));
  }
}

inline int grid_rows(int64_t items, int64_t per_cta, int ctas_per_sm, int sms) {
  int64_t need = (items + per_cta - 1) / per_cta;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)ctas_per_sm * sms;
  return (int)(need < cap ? need : cap);
}

// class-wide sum kinds through the tile kernel (2 <= C <= 32 classes, the tile and >= 2 stages fit in shared memory)
cudaError_t try_launch_agg_class_tile(const AggArgs& a, const FinArgs& f0, int sms, cudaStream_t st, bool* launched) {
  *launched = false;
  static const int enabled = [] { const char* e = getenv("SE_AGG_TILE"); return e ? atoi(e) : 1; }();
  if (!enabled || a.M < 1 || a.n < 1 || a.n >= (int64_t)0x7fffff00) return cudaSuccess;
  // one warp per CTA (128-row tiles), one stage: shared memory bounds occupancy and what counts is the number of
  // boxes in flight per SM (measured, boosting-real M=10 K=26: 1 warp x 1 stage 2.75 ms, 2 warps x 1 stage 2.78,
  // 2 warps x 2 stages 4.32, 2 warps x 4 stages 8.59; streaming path 3.01)
  constexpr int warps = 1;
  const int kAT = 32 * warps, kAR = 128 * warps;
  ClassTileArgs ta{};
  FinArgs f = f0;
  ta.M = a.M;
  switch (a.kind) {
    case SE_AGG_GBM_CLASSIFIER:
      if (a.dim < 2) return cudaSuccess;  // binary dim-1 form: two outputs from one sum (streaming path)
      ta.C = a.dim; ta.a = a.weights; ta.init = a.init; break;
    case SE_AGG_BAGGING_SOFT: ta.C = a.K; break;
    case SE_AGG_BOOSTING_REAL: ta.C = a.K; ta.logp = 1; break;
    default: return cudaSuccess;
  }
  const int C = ta.C;
  if (C < 2 || C > 32) return cudaSuccess;
  f.C = C;
  ta.G = 32 / C;
  if (ta.G > a.M) ta.G = a.M;
  if (ta.G > 8) ta.G = 8;
  const int box_rows = ta.G * C;
  const size_t stage_bytes = (size_t)box_rows * kAR * sizeof(float);
  const size_t total_bytes = (size_t)C * kAR * sizeof(float);
  static const int forced_stages = [] { const char* e = getenv("SE_AGG_TILE_STAGES"); return e ? atoi(e) : 0; }();
  const int stages = forced_stages >= 1 && forced_stages <= kAggMaxStages ? forced_stages : 1;
  const size_t smem = total_bytes + stages * stage_bytes + 128;
  ta.stages = stages;
  CUtensorMap mapP;
  cudaError_t e = make_tile_map_rows(&mapP, a.P, a.n, a.ld, (int64_t)a.M * C, kAR, box_rows);
  if (e != cudaSuccess) return e;
  int per_sm = (int)((228 * 1024) / (smem + 1280));
  if (per_sm > 16) per_sm = 16;
  if (per_sm < 1) return cudaSuccess;
  const int64_t ntiles = (a.n + kAR - 1) / kAR;
  const int64_t cap = (int64_t)per_sm * sms;
  const int grid = (int)(ntiles < cap ? ntiles : cap);
#define SE_CT(CM)                                                                                        \
  {                                                                                                      \
    auto kern = agg_class_tile_kernel<CM, warps>;                                                        \
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
    if (e != cudaSuccess) return e;                                                                      \
    kern<<<grid, kAT, smem, st>>>(ta, f, mapP);                                                          \
  }
  if (C <= 4) SE_CT(4) else if (C <= 8) SE_CT(8) else if (C <= 16) SE_CT(16) else SE_CT(32)
#undef SE_CT
  *launched = true;
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_agg(const AggArgs& a, int ctas_per_sm, int sms, cudaStream_t st) {
  const int grid4 = grid_rows(a.n >> 2, kBlock, ctas_per_sm, sms);
  const int grid1 = grid_rows(a.n, kBlock, ctas_per_sm, sms);
  FinArgs f{};
  f.kind = a.kind; f.K = a.K; f.dim = a.dim; f.loss = a.loss; f.M = a.M;
  f.n = a.n; f.ld = a.ld_out; f.raw = a.raw; f.prob = a.prob; f.label = a.label;
  f.bad_label = a.bad_label;
  f.inv_km1 = 1.0 / (double)((a.K > 1 ? a.K : 2) - 1);
  f.sum_a = 0.0;
  {
    bool launched = false;
    const cudaError_t e = try_launch_agg_class_tile(a, f, sms, st, &launched);
    if (e != cudaSuccess || launched) return e;
  }
  switch (a.kind) {
    case SE_AGG_GBM_REGRESSOR:
      agg_sum_kernel<false><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, 1, a.weights, a.init,
                                                       nullptr, 0.f, a.raw, a.ld_out);
      return cudaGetLastError();
    case SE_AGG_BAGGING_REGRESSOR:
      agg_sum_kernel<false><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, 1, nullptr, nullptr,
                                                       nullptr, (float)a.M, a.raw, a.ld_out);
      return cudaGetLastError();
    case SE_AGG_BOOSTING_REG_MEAN:  // dot(predictions, weights) / Σ weights  (BoostingRegressor.scala:339-342)
      agg_sum_kernel<false><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, 1, a.weights, nullptr,
                                                       nullptr, (float)a.sum_weights, a.raw, a.ld_out);
      return cudaGetLastError();
    case SE_AGG_BOOSTING_REG_MEDIAN: {
      if (a.M < 1) return cudaErrorInvalidValue;
      int Mp = 1;
      while (Mp < a.M) Mp <<= 1;
      if (Mp <= 64 && a.n > 0 && a.n < (int64_t)0x7fffff00) {  // registers, tiles prefetched by TMA
        CUtensorMap mapP;
        cudaError_t e = make_tile_map(&mapP, a.P, a.n, a.ld, a.M, 128);
        if (e != cudaSuccess) return e;
        const size_t smem = 2 * (size_t)a.M * 128 * sizeof(float) + (size_t)a.M * sizeof(double) + 128;
        const int grid = grid_rows(a.n, 128, 8, sms);
        if (a.wm_mode != 0 && a.weights64_host != nullptr && (a.wm_mode == 2 || (a.wm_list != nullptr && a.wm_count != nullptr))) {
          // fast path: keys-only sort + model-order sums; rows inside the rounding margin go to the exact list kernel
          WmWeights wts;
          double total = 0.0, tau = 0.0;
          wm_fast_operands(a.weights64_host, a.M, a.wm_mode, &wts, &total, &tau);
          const bool margin = (a.wm_mode == 1);
          const size_t fsmem = 2 * (size_t)a.M * 128 * sizeof(float) + 128;
          if (margin) {
            e = cudaMemsetAsync(a.wm_count, 0, sizeof(unsigned int), st);
            if (e != cudaSuccess) return e;
          }
          switch (Mp) {
#define SE_WMF(MPV)                                                                                             \
  case MPV: {                                                                                                   \
    auto kern = agg_wmedian_fast_kernel<MPV>;                                                                   \
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);                   \
    if (e != cudaSuccess) return e;                                                                             \
    kern<<<grid, 128, fsmem, st>>>(mapP, a.n, a.M, wts, total, tau, margin ? a.wm_list : nullptr, a.wm_count,   \
                                   a.wm_cap, a.raw);                                                            \
    if (margin) agg_wmedian_list_kernel<MPV><<<sms * 4, 128, 0, st>>>(a.P, a.n, a.ld, a.M, a.weights64, a.wm_list, \
                                                                     a.wm_count, a.wm_cap, a.raw);              \
    break;                                                                                                      \
  }
            SE_WMF(1) SE_WMF(2) SE_WMF(4) SE_WMF(8) SE_WMF(16) SE_WMF(32) SE_WMF(64)
#undef SE_WMF
            default: return cudaErrorInvalidValue;
          }
          return cudaGetLastError();
        }
        switch (Mp) {
#define SE_WM(MPV)                                                                                              \
  case MPV: {                                                                                                   \
    auto kern = agg_wmedian_reg_kernel<MPV>;                                                                    \
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                    \
    if (e != cudaSuccess) return e;                                                                             \
    kern<<<grid, 128, smem, st>>>(mapP, a.n, a.M, a.weights64, a.raw);                                          \
    break;                                                                                                      \
  }
          SE_WM(1) SE_WM(2) SE_WM(4) SE_WM(8) SE_WM(16) SE_WM(32) SE_WM(64)
#undef SE_WM
          default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
      }
      const int T = 64;
      const size_t smem = (size_t)a.M * sizeof(double) + (size_t)Mp * T * sizeof(unsigned long long);
      if (smem > 200 * 1024) {  // M > 256: one warp per row
        const size_t wsmem = (size_t)a.M * sizeof(double) + (size_t)kWmWarps * Mp * sizeof(unsigned long long);
        if (wsmem > 200 * 1024) return cudaErrorInvalidValue;  // M > 8192
        if (wsmem > 48 * 1024) {
          cudaError_t e = cudaFuncSetAttribute(agg_wmedian_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem);
          if (e != cudaSuccess) return e;
        }
        int per_sm_w = (int)((220 * 1024) / (wsmem + 1024));
        if (per_sm_w < 1) per_sm_w = 1;
        if (per_sm_w > 16) per_sm_w = 16;
        const int gridw = grid_rows(a.n, kWmWarps, per_sm_w, sms);
        agg_wmedian_warp_kernel<<<gridw, 32 * kWmWarps, wsmem, st>>>(a.P, a.n, a.ld, a.M, Mp, a.weights64, a.raw);
        return cudaGetLastError();
      }
      auto kern = agg_wmedian_kernel<64>;
      if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
      }
      int per_sm = (int)((220 * 1024) / (smem + 1024));
      if (per_sm < 1) per_sm = 1;
      const int grid = grid_rows(a.n, T, per_sm, sms);
      kern<<<grid, T, smem, st>>>(a.P, a.n, a.ld, a.M, Mp, a.weights64, a.raw);
      return cudaGetLastError();
    }
    case SE_AGG_GBM_CLASSIFIER:
      agg_sum_kernel<false><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, a.dim, a.weights, a.init,
                                                       nullptr, 0.f, a.raw, a.ld_out);
      f.C = (a.dim == 1 && a.K == 2) ? 2 : a.dim;
      break;
    case SE_AGG_BAGGING_SOFT:
      agg_sum_kernel<false><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, a.K, nullptr, nullptr,
                                                       nullptr, 0.f, a.raw, a.ld_out);
      f.C = a.K;
      break;
    case SE_AGG_BOOSTING_REAL:
      agg_sum_kernel<true><<<grid4, kBlock, 0, st>>>(a.P, a.n, a.ld, a.M, a.K, nullptr, nullptr,
                                                      nullptr, 0.f, a.raw, a.ld_out);
      f.C = a.K;
      break;
    case SE_AGG_BAGGING_HARD:
    case SE_AGG_BOOSTING_DISCRETE: {
      const bool weighted = (a.kind == SE_AGG_BOOSTING_DISCRETE);
      static const bool packed_ok = [] { const char* e = getenv("SE_VOTES_PACKED"); return !(e && atoi(e) == 0); }();
      if (!weighted && packed_ok && a.M <= 255 && (size_t)((a.K + 3) / 4) * kVR * kBlock * 4 <= 160 * 1024) {
        const size_t psmem = (size_t)((a.K + 3) / 4) * kVR * kBlock * sizeof(uint32_t);
        if (psmem > 48 * 1024) {
          cudaError_t e = cudaFuncSetAttribute(agg_hard_votes_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem);
          if (e != cudaSuccess) return e;
        }
        f.C = a.K;
        const int gridp = grid_rows((a.n + kVR - 1) / kVR, kBlock, ctas_per_sm, sms);
        agg_hard_votes_packed_kernel<<<gridp, kBlock, psmem, st>>>(a.P, a.ld, a.M, f);
        return cudaGetLastError();
      }
      const size_t hsz = weighted ? sizeof(double) : sizeof(float);
      const size_t smem = (size_t)(a.K + 1) * kBlock * hsz + (size_t)a.M * hsz;
      if (smem > 200 * 1024) return cudaErrorInvalidValue;
      auto kern = weighted ? agg_votes_kernel<double> : agg_votes_kernel<float>;
      if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
      }
      f.C = a.K;
      f.sum_a = a.sum_weights;
      kern<<<grid1, kBlock, smem, st>>>(a.P, a.ld, a.M, weighted ? a.weights : nullptr, f);
      return cudaGetLastError();  // epilogue fused: no separate finalize launch
    }
    default: return cudaErrorInvalidValue;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (a.kind == SE_AGG_BOOSTING_DISCRETE) {
    // Σ a_m is needed by the epilogue (host-side sum of the tiny weight vector)
    f.sum_a = a.sum_weights;
  }
  agg_finalize_kernel<<<grid1, kBlock, 0, st>>>(f);
  return cudaGetLastError();
}

cudaError_t launch_agg_finalize(int kind, int C, int K, int dim, int loss, int M, double sum_a, int64_t n, int64_t ld,
                                float* raw, float* prob, float* label, int sms, cudaStream_t st) {
  FinArgs f{};
  f.kind = kind; f.C = C; f.K = K; f.dim = dim; f.loss = loss; f.M = M;
  f.sum_a = sum_a;
  f.n = n; f.ld = ld; f.raw = raw; f.prob = prob; f.label = label;
  f.inv_km1 = 1.0 / (double)((K > 1 ? K : 2) - 1);
  agg_finalize_kernel<<<grid_rows(n, kBlock, 8, sms), kBlock, 0, st>>>(f);
  return cudaGetLastError();
}

}  // namespace se
