// se_wmedian.cuh — the weighted median's per-row building blocks (ensemble/Utils.scala:26-40), shared by the
// aggregation kernels of se_agg.cu (members' outputs in SE_SLOT_P) and the one-pass forest kernel of se_models.cu
// (members' leaves parked in shared memory), so both routes select the same element by the same code.
#pragma once
#include <stdint.h>

#include "se_sortnet.h"

namespace se {

// Order-preserving 32-bit key of an fp32 value: unsigned comparison of keys is the float order, -0 and +0 share a key.
__device__ __forceinline__ uint32_t wm_key(float x) {
  const uint32_t u = __float_as_uint(x + 0.0f);  // -0 -> +0: equal values stay ties
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float wm_unkey(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// sort of the (key, model) words + the reference's sorted-order cumulative sums (ensemble/Utils.scala:31-38)
template <int MP>
__device__ __forceinline__ unsigned long long wm_exact_pick(unsigned long long (&w)[MP], int M, const double* s_a) {
  sortnet_oddeven<MP>(w, [](unsigned long long& x, unsigned long long& y) {
    const bool swap = x > y;
    const unsigned long long lo = swap ? y : x, hi = swap ? x : y;
    x = lo;
    y = hi;
  });
  double total = 0.0;
#pragma unroll
  for (int m = 0; m < MP; ++m)
    if (m < M) total += s_a[(unsigned)w[m]];
  const double half = 0.5 * total;
  double cum = 0.0;
  bool found = false;
  unsigned long long pick = 0ull;
#pragma unroll
  for (int m = 0; m < MP; ++m) {
    if (m < M) {
      cum += s_a[(unsigned)w[m]];
      const bool hit = !found && (cum >= half);
      pick = (hit || (!found && m == M - 1)) ? w[m] : pick;  // last element when nothing reaches half (NaN weights)
      found = found || hit;
    }
  }
  return pick;
}

// ---- weighted median, fast path (M <= 64, all weights finite and >= 0) -------------------------------------------
// The exact pick carries (key, model) words through the sort because the reference accumulates the weights in SORTED
// order (ensemble/Utils.scala:31-38) — 6 ALU-pipe instructions per compare-exchange, and the ALU pipe issues at half
// rate: 4.07 ms for 25 M rows x 32 models.  With weights >= 0 the answer is `the smallest value v whose group-end
// cumulative weight C(v) reaches h = total / 2` (cumulative sums are monotone in fp64 too).  C(v) and h are recursive
// fp64 sums of the same addends as Ĉ(v) = Σ_{x_j <= v} a_j and ĥ = T̂ / 2 taken in MODEL order, so
//     |(C(v) - h) - (Ĉ(v) - ĥ)| <= 3 (M - 1) 2^-53 T (1 + eps)
// and whenever both neighbours of the crossing clear the margin tau = 8 M 2^-53 T̂ the model-order decision IS the
// reference's decision.  So: sort the 32-bit keys alone (min/max, 2 instructions per compare-exchange, Batcher's
// 191-element network), bisect the sorted keys on Ĉ (5 x 32 predicated DADDs with the weights as constant-bank
// operands), and send the rows that do not clear the margin — none for generic weights, the exact ties for
// small-integer weights — to the exact pick (mode 2: all weights equal, where both orders produce the same sums and no
// margin is needed).
struct WmWeights {
  double w[64];
};

// The fast path's kernel operands from the host weights (mode 1: margin, mode 2: equal weights, no margin): the
// weights padded with zeros to 64, their model-order total (the kernels' own summation order) and the margin tau.
inline void wm_fast_operands(const double* weights, int M, int mode, WmWeights* wts, double* total, double* tau) {
  double s = 0.0;
  for (int m = 0; m < 64; ++m) {
    wts->w[m] = (m < M) ? weights[m] : 0.0;
    s += wts->w[m];  // model order, like the kernels' own sums
  }
  *total = s;
  *tau = (mode == 1) ? 8.0 * (double)M * 1.1102230246251565e-16 * s : -1.0;  // mode 2: every row is safe
}

template <int MP, int L>
__device__ __forceinline__ uint32_t wm_candidate(const uint32_t (&s)[MP], uint32_t t) {
  // level-L bisection probe: position step - 1 + t * 2 * step, t in [0, 2^L) — a select tree over static indices
  constexpr int step = MP >> (L + 1);
  uint32_t v = s[step - 1];
#pragma unroll
  for (int q = 1; q < (1 << L); ++q) v = (t == (uint32_t)q) ? s[step - 1 + q * 2 * step] : v;
  return v;
}

}  // namespace se
