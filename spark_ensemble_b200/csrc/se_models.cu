// se_models.cu — on-device base-model evaluation over the column-major feature matrix X[d][n].
//
// The reference obtains the direction h (GBMRegressor.scala:405,435), class probabilities and
// predictions (BoostingClassifier.scala:199-200,233) by calling third-party Spark ML
// `model.predict(features)` once per row on the JVM.  Keeping X resident in HBM and evaluating the
// fitted model here means h never crosses PCIe (SURVEY.md §8f-1).  Supported: binary decision trees
// with continuous splits (Spark ContinuousSplit.shouldGoLeft: x <= threshold goes left) and linear
// models.  HasSubBag.slice (ensemble/HasSubBag.scala:81-84) is folded into the feature->column map.
#include <stdlib.h>

#include "se_kernels.h"
#include "se_wmedian.cuh"

namespace se {

namespace {

constexpr int TV = 4;  // rows per thread (one float4 of outputs)

// Outputs of TV consecutive rows whose leaves are node[0..TV): the leaf value (regression / label) or the leaf's
// class-probability vector (one coalesced row store per class).
__device__ __forceinline__ void write_leaf_outputs(const TreeArgs& a, const int (&node)[TV], int64_t i0, const float* s_val) {
  if (s_val == nullptr) {
    for (int k = 0; k < a.n_out; ++k) {
      if (i0 + TV <= a.n) {
        st_stream4(a.out + (int64_t)k * a.ld_out + i0,
                   make_float4(__ldg(a.value + node[0] * a.n_out + k), __ldg(a.value + node[1] * a.n_out + k),
                               __ldg(a.value + node[2] * a.n_out + k), __ldg(a.value + node[3] * a.n_out + k)));
      } else {
#pragma unroll
        for (int e = 0; e < TV; ++e)
          if (i0 + e < a.n) a.out[(int64_t)k * a.ld_out + i0 + e] = __ldg(a.value + node[e] * a.n_out + k);
      }
    }
  } else if (i0 + TV <= a.n) {
    st_stream4(a.out + i0, make_float4(s_val[node[0]], s_val[node[1]], s_val[node[2]], s_val[node[3]]));
  } else {
#pragma unroll
    for (int e = 0; e < TV; ++e)
      if (i0 + e < a.n) a.out[i0 + e] = s_val[node[e]];
  }
}

// Tree arrays are staged once per CTA in shared memory; each thread walks TV rows in lockstep so
// TV independent gathers are in flight.  Rows of a warp are consecutive, so every X access of a
// level is a coalesced 128 B segment per distinct feature.
__global__ void __launch_bounds__(kBlock) tree_predict_kernel(const TreeArgs a) {
  extern __shared__ unsigned char smem_raw[];
  int32_t* s_feat = reinterpret_cast<int32_t*>(smem_raw);
  float* s_thr = reinterpret_cast<float*>(s_feat + a.n_nodes);
  int32_t* s_left = reinterpret_cast<int32_t*>(s_thr + a.n_nodes);
  int32_t* s_right = s_left + a.n_nodes;
  float* s_val = reinterpret_cast<float*>(s_right + a.n_nodes);
  const bool scalar = (a.n_out == 1);
  for (int i = threadIdx.x; i < a.n_nodes; i += kBlock) {
    s_feat[i] = a.feature[i];
    s_thr[i] = a.threshold[i];
    s_left[i] = a.left[i];
    s_right[i] = a.right[i];
    if (scalar) s_val[i] = a.value[i];
  }
  __syncthreads();
  const int64_t ngroups = (a.n + TV - 1) / TV;
  for (int64_t g = (int64_t)blockIdx.x * kBlock + threadIdx.x; g < ngroups;
       g += (int64_t)gridDim.x * kBlock) {
    const int64_t i0 = g * TV;
    int node[TV];
    bool live[TV];
    bool any = false;
#pragma unroll
    for (int e = 0; e < TV; ++e) {
      node[e] = 0;
      live[e] = (i0 + e < a.n) && (s_feat[0] >= 0);
      any |= live[e];
    }
    while (any) {
      float x[TV];
#pragma unroll
      for (int e = 0; e < TV; ++e)
        if (live[e]) x[e] = __ldg(a.X + (int64_t)s_feat[node[e]] * a.ld + i0 + e);
      any = false;
#pragma unroll
      for (int e = 0; e < TV; ++e)
        if (live[e]) {
          node[e] = (x[e] <= s_thr[node[e]]) ? s_left[node[e]] : s_right[node[e]];
          live[e] = s_feat[node[e]] >= 0;
          any |= live[e];
        }
    }
    write_leaf_outputs(a, node, i0, scalar ? s_val : nullptr);
  }
}

// ------------------------------------------------------------------ binned feature matrix (uint8) and its tree walk
// ncu on the fp32 walk above (round 1): 174 B/row of DRAM traffic for a depth-6 tree whose algorithmic need is 24 B/row
// — once the rows of a warp diverge every 4-byte gather drags a whole 32-byte sector (8 rows) in.  Decision trees only
// COMPARE features with thresholds, and Spark's trees draw every threshold of a feature from the <= maxBins - 1 split
// candidates `findSplits` computes once per fit: so X can be replaced, for the walk, by the RANK of each value among the
// thresholds seen so far — bin(x) = #{t : t < x} in a uint8 — and `x <= t_j` becomes `bin(x) <= j`, EXACTLY (no
// rounding involved: it is the same comparison, pre-evaluated).  A gather then costs 1 byte and a sector holds 32 rows:
// 3.5x fewer DRAM bytes for the same walk.  The host side (se_api.cu tree_predict_impl) keeps the per-column threshold
// lists, re-bins the columns a new tree adds thresholds to, and falls back to the fp32 walk when a column would need
// more than 255 thresholds.

// One CTA = one (column, row tile): the column's sorted thresholds sit in shared memory; a thread turns 4 fp32 values
// into 4 ranks (branch-free binary search over <= 255 edges: 8 steps) and stores them as one 32-bit word.
__global__ void __launch_bounds__(kBlock) bin_columns_kernel(const BinArgs a) {
  __shared__ float s_edge[256];
  const int which = blockIdx.y;
  const int col = a.cols[which];
  const int ne = a.n_edges[col];
  for (int i = threadIdx.x; i < 256; i += kBlock) s_edge[i] = (i < ne) ? a.edges[(size_t)col * 256 + i] : INFINITY;
  __syncthreads();
  const float* x = a.X + (int64_t)col * a.ld;
  uint8_t* out = a.X8 + (int64_t)col * a.ld8;
  const int64_t n4 = (a.n + 3) >> 2;  // the slot is padded: a 128-bit read at a 4-aligned row below n stays inside
  for (int64_t g = (int64_t)blockIdx.x * kBlock + threadIdx.x; g < n4; g += (int64_t)gridDim.x * kBlock) {
    const float4 v = ld_stream4(x + 4 * g);
    uint32_t word = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float xv = f4at(v, e);
      // rank = number of edges strictly below xv (NaN ranks 0... Spark sends NaN/missing nowhere: not supported)
      int lo = 0;
#pragma unroll
      for (int step = 128; step > 0; step >>= 1)
        if (lo + step <= 256 && s_edge[lo + step - 1] < xv) lo += step;
      word |= (uint32_t)(lo > 255 ? 255 : lo) << (8 * e);
    }
    *reinterpret_cast<uint32_t*>(out + 4 * g) = word;
  }
}

// Packed node (16 bytes, one 128-bit shared-memory read per row and level): x,y = byte offset of the node's column
// in X8 (column * ld8, 64 bit); z = bin threshold | leaf << 31; w = left | right << 16.
// ncu on the first version (two 8-byte node reads per row and level, 64-bit multiply for the column offset): 39
// instructions per row and level, 45 % issue utilisation at 49 % occupancy — the walk was issue-bound, not DRAM-bound
// (52 % of peak).
template <int W, int MINB>  // W words of 4 consecutive rows per thread (independent gather chains), MINB CTAs per SM
__global__ void __launch_bounds__(kBlock, MINB) tree_predict_binned_kernel(const TreeArgs a, const uint8_t* __restrict__ X8,
                                                                           const uint4* __restrict__ nodes) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* s_node = reinterpret_cast<uint4*>(smem_raw);
  float* s_val = reinterpret_cast<float*>(s_node + a.n_nodes);
  const bool scalar = (a.n_out == 1);
  for (int i = threadIdx.x; i < a.n_nodes; i += kBlock) {
    s_node[i] = nodes[i];
    if (scalar) s_val[i] = a.value[i];
  }
  __syncthreads();
  const int64_t ngroups = (a.n + TV - 1) / TV;          // groups of 4 rows
  const int64_t nsuper = (ngroups + W - 1) / W;         // a thread owns W groups, kBlock apart inside a CTA tile
  for (int64_t sg = blockIdx.x; sg * kBlock < nsuper * kBlock && sg * (int64_t)kBlock * W < ngroups; sg += gridDim.x) {
    int node[W][TV];
    int64_t i0[W];
    bool done[W];
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const int64_t g = (sg * W + w) * kBlock + threadIdx.x;   // coalesced: consecutive threads, consecutive groups
      i0[w] = g * TV;
      done[w] = g >= ngroups;
#pragma unroll
      for (int e = 0; e < TV; ++e) node[w][e] = 0;
    }
    for (;;) {
      bool any = false;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        if (done[w]) continue;
        const bool full = (i0[w] + TV <= a.n);
        const uint8_t* row = X8 + i0[w];
        uint4 nd[TV];
        bool live[TV];
        bool anyw = false;
#pragma unroll
        for (int e = 0; e < TV; ++e) {
          nd[e] = s_node[node[w][e]];
          live[e] = ((nd[e].z >> 31) == 0) && (full || i0[w] + e < a.n);
          anyw |= live[e];
        }
        if (!anyw) { done[w] = true; continue; }
        any = true;
        uint32_t b[TV];
        // rows of a word that still share a node (always at the root, often below it) are served by ONE 32-bit load
        if (full && node[w][0] == node[w][1] && node[w][1] == node[w][2] && node[w][2] == node[w][3]) {
          const uint64_t off = ((uint64_t)nd[0].y << 32) | nd[0].x;
          const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(row + off));
#pragma unroll
          for (int e = 0; e < TV; ++e) b[e] = (v >> (8 * e)) & 0xFFu;
        } else {
#pragma unroll
          for (int e = 0; e < TV; ++e)
            if (live[e]) b[e] = __ldg(row + ((((uint64_t)nd[e].y) << 32) | nd[e].x) + e);
        }
#pragma unroll
        for (int e = 0; e < TV; ++e)
          if (live[e]) node[w][e] = (b[e] <= (nd[e].z & 0xFFu)) ? (int)(nd[e].w & 0xFFFFu) : (int)(nd[e].w >> 16);
      }
      if (!any) break;
    }
#pragma unroll
    for (int w = 0; w < W; ++w)
      if ((sg * W + w) * kBlock + threadIdx.x < ngroups) write_leaf_outputs(a, node[w], i0[w], scalar ? s_val : nullptr);
  }
}


// ---- shallow trees (<= 64 internal nodes, e.g. depth <= 6): evaluate EVERY node's comparison, then walk in registers.
// The walk above fetches, per 32 consecutive rows, one 32-byte sector per DISTINCT node its rows sit on at each level:
// 1 + 2 + 4 + ... sectors, i.e. about one byte per row and internal node — exactly what reading the node's column for
// every row costs (ncu: 62 B/row for 63 internal nodes).  Same bytes, but here they arrive as fully coalesced,
// INDEPENDENT vector loads (no level-to-level dependency, one wavefront per 128 rows instead of one per sector), four
// byte-compares at a time in SWAR form, and the per-row walk reads its decision bits from shared memory.
//   bit j of a row = rank(x[col_j]) <= t_j; internal node ordinals j are assigned in node order by warp 0.
constexpr int kTreeMaskWords = 4;  // measured at 100 M x 128, depth 6: 1.51 / 1.22 / 1.15 ms for 1 / 2 / 4 words (walk: 1.47)
template <int RW> struct MaskVec;
template <> struct MaskVec<1> { using type = uint32_t; };
template <> struct MaskVec<2> { using type = uint2; };
template <> struct MaskVec<4> { using type = uint4; };

__device__ __forceinline__ uint32_t bytes_le(uint32_t x, uint32_t t, uint32_t t_hi) {
  // bit 7 of every byte lane: x_byte <= t_byte.  Low 7 bits: (t_lo + 128) - x_lo keeps bit 7 iff t_lo >= x_lo (no
  // borrow crosses a lane: every lane of the minuend is >= 128, of the subtrahend <= 127); top bits decide first.
  const uint32_t d = t_hi - (x & 0x7f7f7f7fu);
  return (~x & t) | (~(x ^ t) & d);
}

template <int RW>  // RW words of 4 consecutive rows per thread, fetched as ONE 4*RW-byte load per node
__global__ void __launch_bounds__(kBlock, 4) tree_predict_mask_kernel(const TreeArgs a, const uint8_t* __restrict__ X8,
                                                                      const uint4* __restrict__ nodes) {
  using V = typename MaskVec<RW>::type;
  __shared__ unsigned long long s_off[64];
  __shared__ uint32_t s_thr[64];
  __shared__ uint32_t s_walk[256];  // ordinal | left << 8 | right << 16 | leaf << 31
  __shared__ float s_val[256];
  __shared__ __align__(16) uint32_t s_acc[8][kBlock * RW];  // [8 nodes per byte][thread][word]: byte e = row e of the word
  __shared__ int s_i8;
  const int tid = threadIdx.x, lane = tid & 31;
  const bool scalar = (a.n_out == 1);
  if (tid < 32) {
    int base = 0;
    for (int c = 0; c < a.n_nodes; c += 32) {
      const int i = c + lane;
      const uint4 nd = (i < a.n_nodes) ? nodes[i] : make_uint4(0u, 0u, 0x80000000u, 0u);
      const bool internal = (nd.z >> 31) == 0;
      const unsigned m = __ballot_sync(0xffffffffu, internal);
      const int ord = base + __popc(m & ((1u << lane) - 1u));
      if (i < a.n_nodes) {
        s_walk[i] = internal ? ((uint32_t)ord | ((nd.w & 0xFFu) << 8) | (((nd.w >> 16) & 0xFFu) << 16)) : 0x80000000u;
        if (internal) {
          s_off[ord] = ((unsigned long long)nd.y << 32) | nd.x;
          s_thr[ord] = (nd.z & 0xFFu) * 0x01010101u;
        }
      }
      base += __popc(m);
    }
    __syncwarp();
    const int i8 = (base + 7) & ~7;  // padded with repeats of node 0's column (their bits are never read)
    for (int j = base + lane; j < i8; j += 32) {
      s_off[j] = s_off[0];
      s_thr[j] = 0u;
    }
    if (lane == 0) s_i8 = i8;
  }
  if (scalar)
    for (int i = tid; i < a.n_nodes; i += kBlock) s_val[i] = a.value[i];
  __syncthreads();
  const int i8 = s_i8;
  constexpr int RPT = 4 * RW;
  const int64_t ngroups = (a.n + RPT - 1) / RPT;
  const unsigned char* my = reinterpret_cast<const unsigned char*>(&s_acc[0][tid * RW]);
  constexpr int kPlane = kBlock * RW * 4;  // bytes between the planes of s_acc
  for (int64_t g = (int64_t)blockIdx.x * kBlock + tid; g < ngroups; g += (int64_t)gridDim.x * kBlock) {
    const int64_t r0 = g * RPT;  // X8 columns are padded to 128 rows: the vector load stays inside the column
    const uint8_t* row = X8 + r0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (8 * k >= i8) break;
      uint32_t acc[RW];
#pragma unroll
      for (int w = 0; w < RW; ++w) acc[w] = 0u;
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const int j = 8 * k + s;
        const uint32_t t = s_thr[j];
        const V v = __ldg(reinterpret_cast<const V*>(row + s_off[j]));
        const uint32_t* xs = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int w = 0; w < RW; ++w) {
          const uint32_t le = bytes_le(xs[w], t, t | 0x80808080u);
          acc[w] |= (s == 7 ? le : (le >> (7 - s))) & (0x01010101u << s);
        }
      }
      *reinterpret_cast<V*>(&s_acc[k][tid * RW]) = *reinterpret_cast<const V*>(acc);
    }
    // the thread reads back only what it stored itself: no barrier
#pragma unroll
    for (int w = 0; w < RW; ++w) {
      if (r0 + 4 * w >= a.n) break;
      int node[TV];
      uint32_t wk[TV];
#pragma unroll
      for (int e = 0; e < TV; ++e) node[e] = 0, wk[e] = s_walk[0];
      for (;;) {
        bool any = false;
#pragma unroll
        for (int e = 0; e < TV; ++e) {
          if (wk[e] >> 31) continue;
          any = true;
          const uint32_t ord = wk[e] & 0xFFu;
          const uint32_t bits = my[(ord >> 3) * kPlane + 4 * w + e];
          node[e] = (int)(((bits >> (ord & 7u)) & 1u) ? (wk[e] >> 8) & 0xFFu : (wk[e] >> 16) & 0xFFu);
          wk[e] = s_walk[node[e]];
        }
        if (!any) break;
      }
      write_leaf_outputs(a, node, r0 + 4 * w, scalar ? s_val : nullptr);
    }
  }
}


// ---- a forest in one pass -----------------------------------------------------------------------------------------
// transform() of a tree ensemble evaluated tree by tree reads each tree's columns of the rank matrix again (one byte per
// row and internal node, 0.73 ms per depth-5 tree and 100 M rows) and needs an [M][n] prediction array for the
// aggregation kernel.  Here a CTA stages a 256-row tile of the ranks of every column the forest uses in shared memory
// (C x 256 bytes), keeps the packed trees next to it, and every thread walks ALL trees for its row out of shared
// memory, two trees interleaved, accumulating w_t · leaf in fp64 in model order like the reference's loop: the rank
// matrix is read once per chunk of trees and no intermediate is written.
__device__ __forceinline__ void forest_step(const uint2* __restrict__ nodes, const unsigned char* __restrict__ myr, int& nd,
                                            bool& live) {
  const uint2 w = nodes[nd];
  live = (w.x >> 31) == 0;
  if (live) {
    const uint32_t rank = myr[(w.x & 0xFFFFu) * kForestTile];
    nd = (int)((rank <= ((w.x >> 16) & 0xFFu)) ? (w.y & 0xFFFFu) : (w.y >> 16));
  }
}

__global__ void __launch_bounds__(kForestTile) forest_predict_kernel(const ForestArgs a) {
  extern __shared__ __align__(16) unsigned char fsm[];
  for (int i = threadIdx.x; i < a.blob_bytes / 16; i += kForestTile)
    reinterpret_cast<uint4*>(fsm)[i] = __ldg(reinterpret_cast<const uint4*>(a.blob) + i);
  const double* s_w = reinterpret_cast<const double*>(fsm);
  const unsigned long long* s_coloff = reinterpret_cast<const unsigned long long*>(fsm + a.off_coloff);
  const uint2* s_nodes = reinterpret_cast<const uint2*>(fsm + a.off_nodes);
  const int* s_toff = reinterpret_cast<const int*>(fsm + a.off_treeoff);
  const float* s_val = reinterpret_cast<const float*>(fsm + a.off_values);
  unsigned char* s_rank = fsm + a.off_ranks;
  const int64_t ntiles = (a.n + kForestTile - 1) / kForestTile;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();  // the packed trees are staged (first tile) / the previous tile's walks are over
    const int64_t row0 = tile * kForestTile;
    for (int i = threadIdx.x; i < a.C * (kForestTile / 4); i += kForestTile) {
      const int c = i / (kForestTile / 4), q = i % (kForestTile / 4);
      const int64_t r = row0 + 4 * q;  // columns are padded to 128 rows: a word at r < ld8 stays inside its column
      uint32_t v = 0;
      if (r < a.ld8) v = __ldg(reinterpret_cast<const uint32_t*>(a.X8 + s_coloff[c] + r));
      *reinterpret_cast<uint32_t*>(s_rank + c * kForestTile + 4 * q) = v;
    }
    __syncthreads();
    const int64_t row = row0 + threadIdx.x;
    if (row < a.n) {
      double acc = a.accumulate ? (double)a.out[row] : a.init;
      const unsigned char* myr = s_rank + threadIdx.x;
      int t = 0;
      for (; t + 1 < a.T; t += 2) {  // two independent walks in flight
        const uint2* n0 = s_nodes + s_toff[t];
        const uint2* n1 = s_nodes + s_toff[t + 1];
        int d0 = 0, d1 = 0;
        bool l0 = true, l1 = true;
        while (l0 || l1) {
          if (l0) forest_step(n0, myr, d0, l0);
          if (l1) forest_step(n1, myr, d1, l1);
        }
        acc += s_w[t] * (double)s_val[s_toff[t] + d0];  // model order (GBMRegressor.scala:534-537)
        acc += s_w[t + 1] * (double)s_val[s_toff[t + 1] + d1];
      }
      if (t < a.T) {
        const uint2* n0 = s_nodes + s_toff[t];
        int d0 = 0;
        bool l0 = true;
        while (l0) forest_step(n0, myr, d0, l0);
        acc += s_w[t] * (double)s_val[s_toff[t] + d0];
      }
      a.out[row] = (float)acc;
    }
  }
}

// The same tile for classifier ensembles.  Phase 1: every thread walks every tree of the chunk for its row (two walks
// in flight) and parks the leaf's ordinal — or, for label leaves, the label itself — in shared memory, [T][256] uint16.
// Phase 2: the classes are swept kClassGroup at a time with fp64 accumulators in registers, each adding the trees in
// model order (the reference's loop order), and every class sum leaves as one coalesced row store into RAW[c].  Class
// probabilities come from the leaf table in global memory (K floats per leaf: L1/L2-resident for realistic forests),
// so neither K nor the class range of a chunk costs shared memory.
constexpr int kClassGroup = 4;

template <int MODE>
__global__ void __launch_bounds__(kForestTile, 2) forest_classify_kernel(const ForestClassArgs a) {
  extern __shared__ __align__(16) unsigned char fsm[];
  for (int i = threadIdx.x; i < a.blob_bytes / 16; i += kForestTile)
    reinterpret_cast<uint4*>(fsm)[i] = __ldg(reinterpret_cast<const uint4*>(a.blob) + i);
  const double* s_w = reinterpret_cast<const double*>(fsm);
  const double* s_init = reinterpret_cast<const double*>(fsm + a.off_init);
  const unsigned long long* s_coloff = reinterpret_cast<const unsigned long long*>(fsm + a.off_coloff);
  const uint2* s_nodes = reinterpret_cast<const uint2*>(fsm + a.off_nodes);
  const int* s_toff = reinterpret_cast<const int*>(fsm + a.off_treeoff);
  const int* s_lbase = reinterpret_cast<const int*>(fsm + a.off_lbase);
  const int* s_cstart = reinterpret_cast<const int*>(fsm + a.off_cstart);
  unsigned char* s_rank = fsm + a.off_ranks;
  uint16_t* s_park = reinterpret_cast<uint16_t*>(fsm + a.off_parked) + threadIdx.x;  // this thread's column
  const int64_t ntiles = (a.n + kForestTile - 1) / kForestTile;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();  // the packed trees are staged (first tile) / the previous tile's ranks are no longer read
    const int64_t row0 = tile * kForestTile;
    for (int i = threadIdx.x; i < a.C * (kForestTile / 4); i += kForestTile) {
      const int c = i / (kForestTile / 4), q = i % (kForestTile / 4);
      const int64_t r = row0 + 4 * q;  // columns are padded to 128 rows: a word at r < ld8 stays inside its column
      uint32_t v = 0;
      if (r < a.ld8) v = __ldg(reinterpret_cast<const uint32_t*>(a.X8 + s_coloff[c] + r));
      *reinterpret_cast<uint32_t*>(s_rank + c * kForestTile + 4 * q) = v;
    }
    __syncthreads();
    const int64_t row = row0 + threadIdx.x;
    if (row >= a.n) continue;  // no barrier below: a thread only reads back what it parked itself
    const unsigned char* myr = s_rank + threadIdx.x;
    auto park = [&](int t, int d) {
      const uint32_t ord = s_nodes[s_toff[t] + d].y;
      s_park[t * kForestTile] =
          (MODE == kForestLabelLeaves) ? (uint16_t)__float2uint_rz(__ldg(a.leaves + s_lbase[t] + ord)) : (uint16_t)ord;
    };
    int t = 0;
    for (; t + 1 < a.T; t += 2) {  // two independent walks in flight
      const uint2* n0 = s_nodes + s_toff[t];
      const uint2* n1 = s_nodes + s_toff[t + 1];
      int d0 = 0, d1 = 0;
      bool l0 = true, l1 = true;
      while (l0 || l1) {
        if (l0) forest_step(n0, myr, d0, l0);
        if (l1) forest_step(n1, myr, d1, l1);
      }
      park(t, d0);
      park(t + 1, d1);
    }
    if (t < a.T) {
      int d0 = 0;
      bool l0 = true;
      while (l0) forest_step(s_nodes + s_toff[t], myr, d0, l0);
      park(t, d0);
    }
    float* out = a.raw + row;
    if (MODE == kForestScalarLeaves) {  // GBM: class c sums its own trees, init_c + Σ_i a_ic · tree_ic(x)
      for (int c = a.c0; c < a.c1; ++c) {
        double acc = (c >= a.acc0 && c < a.acc1) ? (double)out[(int64_t)c * a.ld_raw] : s_init[c - a.c0];
        for (int u = s_cstart[c - a.c0]; u < s_cstart[c - a.c0 + 1]; ++u)
          acc += s_w[u] * (double)__ldg(a.leaves + s_lbase[u] + s_park[u * kForestTile]);
        out[(int64_t)c * a.ld_raw] = (float)acc;
      }
    } else {
      for (int c = a.c0; c < a.c1; c += kClassGroup) {
        double acc[kClassGroup];
#pragma unroll
        for (int j = 0; j < kClassGroup; ++j)
          acc[j] = (c + j < a.c1 && c + j >= a.acc0 && c + j < a.acc1) ? (double)out[(int64_t)(c + j) * a.ld_raw] : 0.0;
        for (int u = 0; u < a.T; ++u) {
          const int v = s_park[u * kForestTile];
          if (MODE == kForestLabelLeaves) {  // a vote of weight w_u for class v
#pragma unroll
            for (int j = 0; j < kClassGroup; ++j) acc[j] += (v == c + j) ? s_w[u] : 0.0;
          } else {  // the leaf's class vector, this group's slice
            const float* lv = a.leaves + s_lbase[u] + (int64_t)v * a.K + c;
#pragma unroll
            for (int j = 0; j < kClassGroup; ++j)
              if (c + j < a.c1) acc[j] += s_w[u] * (double)__ldg(lv + j);
          }
        }
#pragma unroll
        for (int j = 0; j < kClassGroup; ++j)
          if (c + j < a.c1) out[(int64_t)(c + j) * a.ld_raw] = (float)acc[j];
      }
    }
  }
}

// The same tile for the weighted median of the members (AdaBoost.R2, votingStrategy "median").  The median needs all
// T leaf values of a row at once, so phase 1 parks each tree's leaf as its order-preserving 32-bit key (wm_key) in the
// thread's own column of shared memory, [T][256], and phase 2 selects from them in registers with the aggregation's
// own per-row code (se_wmedian.cuh): the keys-only sort and model-order bisection of the fast path, and the exact
// (key, model) pick for mode 0 and for the rows whose decision lies inside the rounding margin.  The exact pick runs
// in the same thread from the parked keys, so no row list and no second pass over the ranks exist; it reloads the
// keys rather than keeping them, so the fast path's keys and the exact pick's words are never live together.  At
// MP = 64 the bisection reads the model-order keys from the parked column in a rolled loop instead of a second
// register copy: with both 64-key copies in registers (agg_wmedian_fast_kernel: 246) this kernel spilled; so it uses
// 207 registers and no local memory.
template <int MP>
__global__ void __launch_bounds__(kForestTile, (MP >= 32) ? 1 : 2)
    forest_wmedian_kernel(const ForestWmArgs a, const __grid_constant__ WmWeights wts, const double total, const double tau) {
  extern __shared__ __align__(16) unsigned char fsm[];
  for (int i = threadIdx.x; i < a.blob_bytes / 16; i += kForestTile)
    reinterpret_cast<uint4*>(fsm)[i] = __ldg(reinterpret_cast<const uint4*>(a.blob) + i);
  const double* s_w = reinterpret_cast<const double*>(fsm);
  const unsigned long long* s_coloff = reinterpret_cast<const unsigned long long*>(fsm + a.off_coloff);
  const uint2* s_nodes = reinterpret_cast<const uint2*>(fsm + a.off_nodes);
  const int* s_toff = reinterpret_cast<const int*>(fsm + a.off_treeoff);
  const float* s_val = reinterpret_cast<const float*>(fsm + a.off_values);
  unsigned char* s_rank = fsm + a.off_ranks;
  uint32_t* s_park = reinterpret_cast<uint32_t*>(fsm + a.off_parked) + threadIdx.x;  // this thread's column
  const int M = a.T;
  const double half = 0.5 * total;
  constexpr int LOG = (MP == 1) ? 0 : (MP == 2) ? 1 : (MP == 4) ? 2 : (MP == 8) ? 3 : (MP == 16) ? 4 : (MP == 32) ? 5 : 6;
  const int64_t ntiles = (a.n + kForestTile - 1) / kForestTile;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();  // the packed trees are staged (first tile) / the previous tile's ranks are no longer read
    const int64_t row0 = tile * kForestTile;
    for (int i = threadIdx.x; i < a.C * (kForestTile / 4); i += kForestTile) {
      const int c = i / (kForestTile / 4), q = i % (kForestTile / 4);
      const int64_t r = row0 + 4 * q;  // columns are padded to 128 rows: a word at r < ld8 stays inside its column
      uint32_t v = 0;
      if (r < a.ld8) v = __ldg(reinterpret_cast<const uint32_t*>(a.X8 + s_coloff[c] + r));
      *reinterpret_cast<uint32_t*>(s_rank + c * kForestTile + 4 * q) = v;
    }
    __syncthreads();
    const int64_t row = row0 + threadIdx.x;
    if (row >= a.n) continue;  // no barrier or warp collective below: a thread only reads back what it parked itself
    const unsigned char* myr = s_rank + threadIdx.x;
    int t = 0;
    for (; t + 1 < M; t += 2) {  // two independent walks in flight
      const uint2* n0 = s_nodes + s_toff[t];
      const uint2* n1 = s_nodes + s_toff[t + 1];
      int d0 = 0, d1 = 0;
      bool l0 = true, l1 = true;
      while (l0 || l1) {
        if (l0) forest_step(n0, myr, d0, l0);
        if (l1) forest_step(n1, myr, d1, l1);
      }
      s_park[t * kForestTile] = wm_key(s_val[s_toff[t] + d0]);
      s_park[(t + 1) * kForestTile] = wm_key(s_val[s_toff[t + 1] + d1]);
    }
    if (t < M) {
      int d0 = 0;
      bool l0 = true;
      while (l0) forest_step(s_nodes + s_toff[t], myr, d0, l0);
      s_park[t * kForestTile] = wm_key(s_val[s_toff[t] + d0]);
    }
    auto leaf_key = [&](int m) { return s_park[m * kForestTile]; };
    constexpr bool kRegKeys = MP < 64;  // model-order keys in registers, or read back from the parked column
    bool exact = a.wm_mode == 0;
    uint32_t v_hi = 0;
    if (!exact) {  // the fast path of agg_wmedian_fast_kernel, row for row
      uint32_t key[kRegKeys ? MP : 1], s[MP];
#pragma unroll
      for (int m = 0; m < MP; ++m) {
        s[m] = 0xFFFFFFFFu;  // padding sorts last and carries weight 0
        if (m < M) s[m] = leaf_key(m);
        if constexpr (kRegKeys) key[m] = s[m];
      }
      sortnet_oddeven<MP>(s, [](uint32_t& x, uint32_t& y) {
        const uint32_t lo = min(x, y), hi = max(x, y);
        x = lo;
        y = hi;
      });
      // invariant: P(lo) false, P(hi) true with P(k) := Ĉ(s[k]) >= ĥ; lo = t - 1, hi = t after LOG probes
      uint32_t tt = 0;
      v_hi = s[MP - 1];
      double c_lo = 0.0, c_hi = total;
      auto probe = [&](uint32_t v) {
        double c = 0.0;
        if constexpr (kRegKeys) {
#pragma unroll
          for (int m = 0; m < MP; ++m) {
            const double b = __hiloint2double((key[m] <= v) ? 0x3ff00000 : 0, 0);
            c = fma(wts.w[m], b, c);
          }
        } else {  // a rolled loop over the parked column: weights by index from the parameter bank (m >= M: weight 0)
#pragma unroll 4
          for (int m = 0; m < M; ++m) {
            const double b = __hiloint2double((leaf_key(m) <= v) ? 0x3ff00000 : 0, 0);
            c = fma(wts.w[m], b, c);
          }
        }
        const bool right = !(c >= half);
        c_lo = right ? c : c_lo;
        c_hi = right ? c_hi : c;
        v_hi = right ? v_hi : v;
        tt = 2u * tt + (right ? 1u : 0u);
      };
      if constexpr (LOG > 0) probe(wm_candidate<MP, 0>(s, tt));
      if constexpr (LOG > 1) probe(wm_candidate<MP, 1>(s, tt));
      if constexpr (LOG > 2) probe(wm_candidate<MP, 2>(s, tt));
      if constexpr (LOG > 3) probe(wm_candidate<MP, 3>(s, tt));
      if constexpr (LOG > 4) probe(wm_candidate<MP, 4>(s, tt));
      if constexpr (LOG > 5) probe(wm_candidate<MP, 5>(s, tt));
      const bool safe = (c_hi - half > tau) && (half - c_lo > tau);
      if (a.wm_mode == 1 && !safe) {  // the decision could depend on the order of summation
        exact = true;
        atomicAdd(a.deferred, 1u);
      }
    }
    if (exact) {
      unsigned long long w[MP];
#pragma unroll
      for (int m = 0; m < MP; ++m) {
        w[m] = ~0ull;  // padding sorts last
        if (m < M) w[m] = ((unsigned long long)leaf_key(m) << 32) | (unsigned long long)(unsigned)m;
      }
      v_hi = (uint32_t)(wm_exact_pick<MP>(w, M, s_w) >> 32);
    }
    a.out[row] = wm_unkey(v_hi);
  }
}

constexpr int LU = 8;

__global__ void __launch_bounds__(kBlock) linear_predict_kernel(const float* __restrict__ X, int64_t n,
                                                               int64_t ld, int n_coef,
                                                               const float* __restrict__ coef,
                                                               const int32_t* __restrict__ cols,
                                                               float intercept, float* __restrict__ out) {
  const int64_t n4 = n >> 2;
  for (int64_t g = (int64_t)blockIdx.x * kBlock + threadIdx.x; g < n4;
       g += (int64_t)gridDim.x * kBlock) {
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
    for (int j0 = 0; j0 < n_coef; j0 += LU) {
      float4 v[LU];
      float c[LU];
#pragma unroll
      for (int u = 0; u < LU; ++u)
        if (j0 + u < n_coef) {
          const int64_t col = cols ? cols[j0 + u] : (j0 + u);
          v[u] = ld_stream4(X + col * ld + 4 * g);
          c[u] = coef[j0 + u];
        }
#pragma unroll
      for (int u = 0; u < LU; ++u)
        if (j0 + u < n_coef) {
          float4& s = (u & 1) ? s1 : s0;
          s.x = fmaf(c[u], v[u].x, s.x); s.y = fmaf(c[u], v[u].y, s.y);
          s.z = fmaf(c[u], v[u].z, s.z); s.w = fmaf(c[u], v[u].w, s.w);
        }
    }
    st_stream4(out + 4 * g, make_float4(intercept + (s0.x + s1.x), intercept + (s0.y + s1.y),
                                        intercept + (s0.z + s1.z), intercept + (s0.w + s1.w)));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    float s = 0.f;
    for (int j = 0; j < n_coef; ++j) {
      const int64_t col = cols ? cols[j] : j;
      s = fmaf(coef[j], X[col * ld + i], s);
    }
    out[i] = intercept + s;
  }
}

}  // namespace

cudaError_t launch_tree_predict(const TreeArgs& a, int sms, cudaStream_t st) {
  const size_t smem = (size_t)a.n_nodes * 5 * sizeof(float);
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(tree_predict_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const int64_t ngroups = (a.n + TV - 1) / TV;
  int64_t need = (ngroups + kBlock - 1) / kBlock;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)sms * 8;
  tree_predict_kernel<<<(int)(need < cap ? need : cap), kBlock, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_bin_columns(const BinArgs& a, int n_cols, int sms, cudaStream_t st) {
  if (n_cols <= 0) return cudaSuccess;
  const int64_t n4 = (a.n + 3) >> 2;
  int64_t gx = (n4 + kBlock - 1) / kBlock;
  const int64_t cap = ((int64_t)sms * 16 + n_cols - 1) / n_cols;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  bin_columns_kernel<<<dim3((unsigned)gx, (unsigned)n_cols), kBlock, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_tree_predict_binned(const TreeArgs& a, const uint8_t* X8, const uint4* nodes, int n_internal, int mask_mode,
                                       int sms, cudaStream_t st) {
  const size_t smem = (size_t)a.n_nodes * (sizeof(uint4) + sizeof(float));
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  static const int variant = [] { const char* e = getenv("SE_TREE_VARIANT"); return e ? atoi(e) : 0; }();
  const int64_t ngroups = (a.n + TV - 1) / TV;
  // shallow trees: all node comparisons from coalesced column reads, then a walk over bits (tree_predict_mask_kernel)
  // SE_TREE_VARIANT: 0 default, 1-5 and 9 walk variants, 10/11/12 all-nodes kernel with 1/2/4 words per thread
  if (mask_mode && n_internal <= 64 && a.n_nodes <= 256 && (variant == 0 || variant >= 10)) {
    const int rw = variant == 10 ? 1 : variant == 11 ? 2 : variant == 12 ? 4 : kTreeMaskWords;
    const int64_t need0 = (a.n + 4 * rw - 1) / (4 * rw);
    int64_t need = (need0 + kBlock - 1) / kBlock;
    if (need < 1) need = 1;
    const int64_t cap = (int64_t)sms * 16;
    const int grid = (int)(need < cap ? need : cap);
    if (rw == 1) tree_predict_mask_kernel<1><<<grid, kBlock, 0, st>>>(a, X8, nodes);
    else if (rw == 2) tree_predict_mask_kernel<2><<<grid, kBlock, 0, st>>>(a, X8, nodes);
    else tree_predict_mask_kernel<4><<<grid, kBlock, 0, st>>>(a, X8, nodes);
    return cudaGetLastError();
  }
#define SE_TREE_LAUNCH(W, MINB)                                                                                      \
  do {                                                                                                               \
    auto kern = tree_predict_binned_kernel<W, MINB>;                                                                 \
    if (smem > 48 * 1024) {                                                                                          \
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
      if (e != cudaSuccess) return e;                                                                                \
    }                                                                                                                \
    int64_t need = (ngroups + (int64_t)kBlock * W - 1) / ((int64_t)kBlock * W);                                      \
    if (need < 1) need = 1;                                                                                          \
    const int64_t cap = (int64_t)sms * 16;                                                                           \
    kern<<<(int)(need < cap ? need : cap), kBlock, smem, st>>>(a, X8, nodes);                                        \
  } while (0)
  switch (variant) {
    case 1: SE_TREE_LAUNCH(1, 8); break;
    case 2: SE_TREE_LAUNCH(2, 4); break;
    case 3: SE_TREE_LAUNCH(2, 3); break;
    case 4: SE_TREE_LAUNCH(4, 2); break;
    case 5: SE_TREE_LAUNCH(1, 6); break;
    default: SE_TREE_LAUNCH(1, 4); break;
  }
#undef SE_TREE_LAUNCH
  return cudaGetLastError();
}

cudaError_t launch_forest_predict(const ForestArgs& a, int sms, cudaStream_t st) {
  const size_t smem = (size_t)a.off_ranks + (size_t)a.C * kForestTile;
  if (a.T < 1 || a.C < 0 || smem > 220 * 1024 || (a.blob_bytes & 15) != 0) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {  // per device and per launch (a handful of launches per transform)
    cudaError_t e = cudaFuncSetAttribute(forest_predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int per_sm = (int)((220 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 8) per_sm = 8;
  int64_t need = (a.n + kForestTile - 1) / kForestTile;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)sms * per_sm;
  forest_predict_kernel<<<(int)(need < cap ? need : cap), kForestTile, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_forest_classify(const ForestClassArgs& a, int sms, cudaStream_t st) {
  const size_t smem = (size_t)a.off_parked + (size_t)a.T * kForestTile * sizeof(uint16_t);
  if (a.T < 1 || a.C < 0 || smem > 220 * 1024 || (a.blob_bytes & 15) != 0 || (a.off_parked & 15) != 0) return cudaErrorInvalidValue;
  auto kern = a.mode == kForestScalarLeaves   ? forest_classify_kernel<kForestScalarLeaves>
              : a.mode == kForestVectorLeaves ? forest_classify_kernel<kForestVectorLeaves>
                                              : forest_classify_kernel<kForestLabelLeaves>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int per_sm = (int)((220 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 8) per_sm = 8;
  int64_t need = (a.n + kForestTile - 1) / kForestTile;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)sms * per_sm;
  kern<<<(int)(need < cap ? need : cap), kForestTile, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_forest_wmedian(const ForestWmArgs& a, int sms, cudaStream_t st) {
  const size_t smem = (size_t)a.off_parked + (size_t)a.T * kForestTile * sizeof(uint32_t);
  if (a.T < 1 || a.T > 64 || a.C < 0 || smem > 220 * 1024 || (a.blob_bytes & 15) != 0 || (a.off_parked & 15) != 0 ||
      (a.wm_mode != 0 && a.weights_host == nullptr) || (a.wm_mode == 1 && a.deferred == nullptr))
    return cudaErrorInvalidValue;
  WmWeights wts;
  double total = 0.0, tau = -1.0;
  if (a.wm_mode != 0) {
    wm_fast_operands(a.weights_host, a.T, a.wm_mode, &wts, &total, &tau);
  } else {
    for (int m = 0; m < 64; ++m) wts.w[m] = 0.0;  // unused: the exact pick reads the blob's weights
  }
  if (a.wm_mode == 1) {
    const cudaError_t e = cudaMemsetAsync(a.deferred, 0, sizeof(unsigned int), st);
    if (e != cudaSuccess) return e;
  }
  int Mp = 1;
  while (Mp < a.T) Mp <<= 1;
  void (*kern)(const ForestWmArgs, const WmWeights, const double, const double) = nullptr;
  switch (Mp) {
    case 1: kern = forest_wmedian_kernel<1>; break;
    case 2: kern = forest_wmedian_kernel<2>; break;
    case 4: kern = forest_wmedian_kernel<4>; break;
    case 8: kern = forest_wmedian_kernel<8>; break;
    case 16: kern = forest_wmedian_kernel<16>; break;
    case 32: kern = forest_wmedian_kernel<32>; break;
    default: kern = forest_wmedian_kernel<64>; break;
  }
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  // resident CTAs per SM from registers and shared memory together
  int per_sm = 1;
  {
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kForestTile, smem);
    if (e != cudaSuccess) return e;
  }
  if (per_sm < 1) per_sm = 1;
  int64_t need = (a.n + kForestTile - 1) / kForestTile;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)sms * per_sm;
  kern<<<(int)(need < cap ? need : cap), kForestTile, smem, st>>>(a, wts, total, tau);
  return cudaGetLastError();
}

cudaError_t launch_linear_predict(const float* X, int64_t n, int64_t ld, int n_coef,
                                  const float* coef, const int32_t* cols, float intercept,
                                  float* out, int sms, cudaStream_t st) {
  int64_t need = ((n >> 2) + kBlock - 1) / kBlock;
  if (need < 1) need = 1;
  const int64_t cap = (int64_t)sms * 8;
  linear_predict_kernel<<<(int)(need < cap ? need : cap), kBlock, 0, st>>>(X, n, ld, n_coef, coef, cols,
                                                                        intercept, out);
  return cudaGetLastError();
}

}  // namespace se
