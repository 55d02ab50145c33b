// SAGPooling for the `GraphSAGE_SAG` / `EAGNN_SAG` variants (SURVEY.md section 8 row f4).
//
// Replaces PyG `SAGPooling(hidden, ratio=0.5, GNN=SAGEConv, aggr='add')` constructed at
// Models/BuckGNN.py:203-208 / 231-236 and applied at :365-367 / :502-504:
//     score = tanh(SAGEConv(hidden, 1, aggr='add')(x, edge_index))          one scalar per node
//     perm  = per-graph top-ceil(ratio * n_g) nodes, descending score        (PyG `topk`)
//     x'    = x[perm] * score[perm],  batch' = batch[perm]
//     edge_index' = edges with both endpoints kept, relabelled, order kept   (PyG `filter_adj`)
//
// Kernels (all deterministic, no floating-point atomics):
//   k_sag_dots        p = x . w_l, q = x . w_r  -- the 512 -> 1 SAGEConv is linear, so
//                     w_l . (sum_j x_j) = sum_j (w_l . x_j): ONE pass over x [N,512] (HBM bound)
//                     and a scalar neighbourhood sum instead of a 512-wide aggregation (x [N,128] for a
//                     hidden_channels = 128 model: the row kernels are templates on the row width)
//   k_sag_score(_big) score_i = tanh(sign * (sum_{j -> i} p_j + b + q_i)) over the CSR keyed by target
//   k_sag_plan        k_g = ceil(ratio * n_g); exclusive scans -> new graph offsets, rank-tile offsets
//   k_sag_sort        graphs of up to 16384 nodes: one CTA per graph sorts 64-bit keys (order-preserving score
//                     bits, descending | local node id) with a bitonic network in shared memory; the first
//                     k_g entries are the kept nodes in PyG's order.  Equal scores keep the lower node id
//                     first = torch.sort(descending, stable)
//   k_sag_rank        larger graphs: rank_i = #{j in graph(i): s_j > s_i or (s_j == s_i and j < i)} by
//                     counting (score tiles broadcast from shared memory); node i is kept iff
//                     rank_i < k_g and lands at row new_ptr[g] + rank_i -- the same order without a sort
//   k_sag_edge_count / k_sag_scan_sums / k_sag_edge_write   order-preserving edge compaction
//   k_gather_rows     out[r] = x[idx[r]] * scale[idx[r]]   (x[perm] * score[perm]; edge rows)
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "aggregate.cuh"
#include "csr_build.cuh"
#include "train.cuh"      // warp_sum

namespace bg {

constexpr int kSagWarps = 8;
constexpr int kRankThreads = 256;
constexpr int kRankPerThread = 4;
constexpr int kRankTileI = kRankThreads * kRankPerThread;   // nodes ranked by one CTA
constexpr int kRankTileJ = 2048;                            // scores staged in shared memory per step
constexpr int kEdgeItemsPerBlock = 4096;                    // 1024 threads x 4 consecutive edges
constexpr int kSagSortMax = 16384;                          // graphs up to this size sort in shared memory (128 KB of keys)

// The four row kernels (k_sag_dots, k_gather_rows, k_sag_bwd_rowdot, k_sag_bwd_dx) are templates on the row width kW:
// 512, or 128 for a hidden_channels = 128 model (the `bg_*128` entry points).  A warp owns a row, each lane
// RowIO<T, kW>::kPer of its columns (train.cuh): 16 interleaved ones at 512, 4 consecutive ones at 128.
template <typename T, int kW>
__global__ void __launch_bounds__(kSagWarps * 32)
k_sag_dots(const T* __restrict__ x, int64_t N, const float* __restrict__ w_l, const float* __restrict__ w_r,
           float* __restrict__ p, float* __restrict__ q) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  float wl[kPer], wr[kPer];
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int c = IO::col_of(lane, i);
    wl[i] = w_l[c];
    wr[i] = w_r[c];
  }
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  for (; r + n_warps < N; r += 2 * n_warps) {                 // two rows in flight per warp
    float v0[kPer], v1[kPer];
    IO::load(x + (size_t)r * kW, lane, v0);
    IO::load(x + (size_t)(r + n_warps) * kW, lane, v1);
    float a0 = 0.f, b0 = 0.f, a1 = 0.f, b1 = 0.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      a0 = fmaf(v0[i], wl[i], a0); b0 = fmaf(v0[i], wr[i], b0);
      a1 = fmaf(v1[i], wl[i], a1); b1 = fmaf(v1[i], wr[i], b1);
    }
    a0 = warp_sum(a0); b0 = warp_sum(b0); a1 = warp_sum(a1); b1 = warp_sum(b1);
    if (lane == 0) { p[r] = a0; q[r] = b0; p[r + n_warps] = a1; q[r + n_warps] = b1; }
  }
  for (; r < N; r += n_warps) {
    float v0[kPer];
    IO::load(x + (size_t)r * kW, lane, v0);
    float a0 = 0.f, b0 = 0.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) { a0 = fmaf(v0[i], wl[i], a0); b0 = fmaf(v0[i], wr[i], b0); }
    a0 = warp_sum(a0); b0 = warp_sum(b0);
    if (lane == 0) { p[r] = a0; q[r] = b0; }
  }
}

// 8 lanes per row (mesh rows have ~5 neighbours); rows above the big-row threshold are left to k_sag_score_big
template <bool kTanh>
__global__ void __launch_bounds__(256)
k_sag_score(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ p,
            const float* __restrict__ q, float bias, float sign, int64_t N, float* __restrict__ score) {
  const int sub = threadIdx.x & 7;
  const int64_t n_groups = ((int64_t)gridDim.x * blockDim.x) >> 3;
  const int64_t n_iter = (N + n_groups - 1) / n_groups;
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  for (int64_t it = 0; it < n_iter; ++it, r += n_groups) {   // uniform trip count: the shuffles below stay convergent
    float s = 0.f;
    bool small = false;
    if (r < N) {
      const int32_t b = rowptr[r], e = rowptr[r + 1];
      small = (e - b) <= kBigRowThreshold;
      if (small)
        for (int32_t i = b + sub; i < e; i += 8) s += p[col[i]];
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (small && sub == 0) score[r] = kTanh ? tanhf(sign * ((s + bias) + q[r])) : s;
  }
}

// one CTA per hub row: strided partial sums, then a fixed-order reduction
template <bool kTanh>
__global__ void __launch_bounds__(256)
k_sag_score_big(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ big_rows,
                const float* __restrict__ p, const float* __restrict__ q, float bias, float sign,
                float* __restrict__ score) {
  __shared__ float red[8];
  const int32_t r = big_rows[blockIdx.x];
  const int32_t b = rowptr[r], e = rowptr[r + 1];
  float s = 0.f;
  for (int32_t i = b + threadIdx.x; i < e; i += 256) s += p[col[i]];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red[w];
    score[r] = kTanh ? tanhf(sign * ((t + bias) + q[r])) : t;
  }
}

// PyG topk: k = ceil(ratio * n) in fp32, as `(ratio * num_nodes.to(torch.float)).ceil()` computes it
BG_DEVINL int32_t sag_keep_count(float ratio, int32_t n) {
  int32_t k = (int32_t)ceilf(ratio * (float)n);
  return min(max(k, 0), n);
}

// single CTA: new_ptr = exclusive scan of k_g, tile_ptr = exclusive scan of ceil(n_g / kRankTileI); info[0] = N'
__global__ void __launch_bounds__(1024)
k_sag_plan(const int32_t* __restrict__ graph_ptr, int32_t G, float ratio, int32_t* __restrict__ new_ptr,
           int32_t* __restrict__ tile_ptr, int32_t* __restrict__ info) {
  __shared__ int32_t sw[32];
  __shared__ int32_t carry_k, carry_t;
  if (threadIdx.x == 0) { carry_k = 0; carry_t = 0; }
  __syncthreads();
  for (int32_t base = 0; base < G; base += 1024) {
    const int32_t g = base + threadIdx.x;
    int32_t k = 0, t = 0;
    if (g < G) {
      const int32_t n = graph_ptr[g + 1] - graph_ptr[g];
      k = sag_keep_count(ratio, n);
      t = (n + kRankTileI - 1) / kRankTileI;
    }
    int32_t tot_k, tot_t;
    const int32_t ex_k = block_exclusive_scan(k, sw, tot_k);
    __syncthreads();
    const int32_t ex_t = block_exclusive_scan(t, sw, tot_t);
    const int32_t ck = carry_k, ct = carry_t;
    if (g < G) { new_ptr[g] = ck + ex_k; tile_ptr[g] = ct + ex_t; }
    __syncthreads();
    if (threadIdx.x == 0) { carry_k = ck + tot_k; carry_t = ct + tot_t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { new_ptr[G] = carry_k; tile_ptr[G] = carry_t; info[0] = carry_k; }
}

// kMode 0: the j range lies wholly before this CTA's nodes (ties count), 1: wholly after (ties do not), 2: overlaps them
template <int kMode>
BG_DEVINL void rank_tile(const float* __restrict__ sj, int32_t cnt, int32_t j_base, const float (&si)[kRankPerThread],
                         const int32_t (&ii)[kRankPerThread], int32_t (&rank)[kRankPerThread]) {
  int32_t jj = 0;
  for (; jj + 4 <= cnt; jj += 4) {
    const float4 s4 = *reinterpret_cast<const float4*>(sj + jj);      // same address in every lane: broadcast
    const float s[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int k = 0; k < kRankPerThread; ++k) {
        if constexpr (kMode == 0) rank[k] += (s[u] >= si[k]) ? 1 : 0;
        else if constexpr (kMode == 1) rank[k] += (s[u] > si[k]) ? 1 : 0;
        else rank[k] += (s[u] > si[k] || (s[u] == si[k] && j_base + jj + u < ii[k])) ? 1 : 0;
      }
    }
  }
  for (; jj < cnt; ++jj) {
    const float s = sj[jj];
#pragma unroll
    for (int k = 0; k < kRankPerThread; ++k) {
      if constexpr (kMode == 0) rank[k] += (s >= si[k]) ? 1 : 0;
      else if constexpr (kMode == 1) rank[k] += (s > si[k]) ? 1 : 0;
      else rank[k] += (s > si[k] || (s == si[k] && j_base + jj < ii[k])) ? 1 : 0;
    }
  }
}

// ascending order of this key = descending score, ties by ascending local node id.  -0.0 is folded onto +0.0 first
// (they compare equal as floats, so a stable float sort does not separate them).
// a NaN score (non-finite activations upstream) ranks as -inf, so both paths still produce a valid permutation: the
// counting rank would otherwise give every NaN rank 0 (all comparisons false) and leave perm slots unwritten
BG_DEVINL float sag_rank_value(float s) { return (s != s) ? -CUDART_INF_F : s; }

BG_DEVINL unsigned long long sag_sort_key(float s, uint32_t local) {
  const uint32_t b = __float_as_uint(sag_rank_value(s) + 0.0f);
  const uint32_t asc = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)(~asc) << 32) | local;
}

// one 1024-thread CTA per graph (grid-stride over graphs); graphs above kSagSortMax nodes are left to k_sag_rank
__global__ void __launch_bounds__(1024)
k_sag_sort(const float* __restrict__ score, const int32_t* __restrict__ graph_ptr, int32_t G,
           const int32_t* __restrict__ new_ptr, int32_t* __restrict__ new_id, int32_t* __restrict__ perm,
           int64_t* __restrict__ batch_out, float* __restrict__ score_out) {
  extern __shared__ unsigned long long sag_keys[];
  for (int32_t g = blockIdx.x; g < G; g += gridDim.x) {
    const int32_t lo = graph_ptr[g], n = graph_ptr[g + 1] - lo;
    if (n <= 0 || n > kSagSortMax) continue;                       // uniform over the CTA
    int32_t P = 1;
    while (P < n) P <<= 1;
    for (int32_t i = threadIdx.x; i < P; i += 1024)
      sag_keys[i] = (i < n) ? sag_sort_key(score[lo + i], (uint32_t)i) : ~0ull;
    __syncthreads();
    for (int32_t k = 2; k <= P; k <<= 1) {
      for (int32_t j = k >> 1; j > 0; j >>= 1) {
        for (int32_t t = threadIdx.x; t < (P >> 1); t += 1024) {
          const int32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));   // bit j clear
          const int32_t l = i | j;
          const unsigned long long a = sag_keys[i], b = sag_keys[l];
          if ((a > b) == ((i & k) == 0)) { sag_keys[i] = b; sag_keys[l] = a; }
        }
        __syncthreads();
      }
    }
    const int32_t base = new_ptr[g], k_g = new_ptr[g + 1] - base;
    for (int32_t r = threadIdx.x; r < n; r += 1024) {
      const int32_t node = lo + (int32_t)(uint32_t)sag_keys[r];
      if (r < k_g) {
        const int32_t nid = base + r;
        new_id[node] = nid;
        perm[nid] = node;
        batch_out[nid] = (int64_t)g;
        score_out[nid] = score[node];
      } else {
        new_id[node] = -1;
      }
    }
    __syncthreads();                                                // the keys are reused by the next graph
  }
}

__global__ void __launch_bounds__(kRankThreads)
k_sag_rank(const float* __restrict__ score, const int32_t* __restrict__ graph_ptr, int32_t G,
           const int32_t* __restrict__ new_ptr, const int32_t* __restrict__ tile_ptr,
           int32_t* __restrict__ new_id, int32_t* __restrict__ perm, int64_t* __restrict__ batch_out,
           float* __restrict__ score_out) {
  __shared__ __align__(16) float sj[kRankTileJ];
  const int32_t t = blockIdx.x;
  if (t >= tile_ptr[G]) return;
  int32_t lo_g = 0, hi_g = G - 1;                 // largest g with tile_ptr[g] <= t (empty graphs own no tile)
  while (lo_g < hi_g) {
    const int32_t mid = (lo_g + hi_g + 1) >> 1;
    if (tile_ptr[mid] <= t) lo_g = mid; else hi_g = mid - 1;
  }
  const int32_t g = lo_g;
  const int32_t lo = graph_ptr[g], hi = graph_ptr[g + 1];
  if (hi - lo <= kSagSortMax) return;             // sorted in shared memory by k_sag_sort
  const int32_t i0 = lo + (t - tile_ptr[g]) * kRankTileI;
  const int32_t i_end = min(i0 + kRankTileI, hi);
  float si[kRankPerThread];
  int32_t ii[kRankPerThread], rank[kRankPerThread];
#pragma unroll
  for (int k = 0; k < kRankPerThread; ++k) {
    ii[k] = i0 + (int32_t)threadIdx.x + k * kRankThreads;
    si[k] = (ii[k] < hi) ? sag_rank_value(score[ii[k]]) : CUDART_INF_F;
    rank[k] = 0;
  }
  for (int32_t jb = lo; jb < hi; jb += kRankTileJ) {
    const int32_t cnt = min(kRankTileJ, hi - jb);
    __syncthreads();
    for (int32_t j = threadIdx.x; j < cnt; j += kRankThreads) sj[j] = sag_rank_value(score[jb + j]);
    __syncthreads();
    // split the staged scores at this CTA's own node range: only the diagonal block needs the index tie-break
    // (i0 - jb and i_end - jb are multiples of kRankTileI or the end of the graph, so the float4 reads stay aligned)
    const int32_t a = max(0, min(cnt, i0 - jb)), b = max(0, min(cnt, i_end - jb));
    if (a > 0) rank_tile<0>(sj, a, jb, si, ii, rank);
    if (b > a) rank_tile<2>(sj + a, b - a, jb + a, si, ii, rank);
    if (cnt > b) rank_tile<1>(sj + b, cnt - b, jb + b, si, ii, rank);
  }
  const int32_t k_g = new_ptr[g + 1] - new_ptr[g];
#pragma unroll
  for (int k = 0; k < kRankPerThread; ++k) {
    if (ii[k] >= hi) continue;
    if (rank[k] < k_g) {
      const int32_t nid = new_ptr[g] + rank[k];
      new_id[ii[k]] = nid;
      perm[nid] = ii[k];
      batch_out[nid] = (int64_t)g;
      score_out[nid] = score[ii[k]];
    } else {
      new_id[ii[k]] = -1;
    }
  }
}

BG_DEVINL bool sag_edge_kept(const int64_t* __restrict__ ei, int64_t E, int64_t N, const int32_t* __restrict__ new_id,
                             int64_t e, int32_t& ns, int32_t& nd) {
  const int64_t s = ei[e], d = ei[E + e];
  if (s < 0 || s >= N || d < 0 || d >= N) return false;
  ns = new_id[s];
  nd = new_id[d];
  return ns >= 0 && nd >= 0;
}

__global__ void __launch_bounds__(1024)
k_sag_edge_count(const int64_t* __restrict__ ei, int64_t E, int64_t N, const int32_t* __restrict__ new_id,
                 int32_t* __restrict__ block_sums) {
  __shared__ int32_t sw[32];
  const int64_t base = (int64_t)blockIdx.x * kEdgeItemsPerBlock + threadIdx.x * 4;
  int32_t s = 0, ns, nd;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (base + i < E && sag_edge_kept(ei, E, N, new_id, base + i, ns, nd)) ++s;
  int32_t total;
  block_exclusive_scan(s, sw, total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single CTA: exclusive scan of the block sums in place; the grand total (E') goes to *total_out
__global__ void __launch_bounds__(1024)
k_sag_scan_sums(int32_t* __restrict__ block_sums, int32_t n_blocks, int32_t* __restrict__ total_out) {
  __shared__ int32_t sw[32];
  __shared__ int32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int32_t base = 0; base < n_blocks; base += 1024) {
    const int32_t i = base + threadIdx.x;
    const int32_t v = (i < n_blocks) ? block_sums[i] : 0;
    int32_t total;
    const int32_t ex = block_exclusive_scan(v, sw, total);
    const int32_t carry = carry_s;
    if (i < n_blocks) block_sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry_s;
}

__global__ void __launch_bounds__(1024)
k_sag_edge_write(const int64_t* __restrict__ ei, int64_t E, int64_t N, const int32_t* __restrict__ new_id,
                 const int32_t* __restrict__ block_offs, int64_t E_out, int64_t* __restrict__ ei_out,
                 int32_t* __restrict__ kept_edge) {
  __shared__ int32_t sw[32];
  const int64_t base = (int64_t)blockIdx.x * kEdgeItemsPerBlock + threadIdx.x * 4;
  int32_t ns[4], nd[4], s = 0;
  bool keep[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    keep[i] = base + i < E && sag_edge_kept(ei, E, N, new_id, base + i, ns[i], nd[i]);
    s += keep[i] ? 1 : 0;
  }
  int32_t total;
  int64_t pos = (int64_t)block_offs[blockIdx.x] + block_exclusive_scan(s, sw, total);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (keep[i] && pos < E_out) {
      ei_out[pos] = ns[i];
      ei_out[E_out + pos] = nd[i];
      if (kept_edge) kept_edge[pos] = (int32_t)(base + i);
      ++pos;
    }
  }
}

// out[r, 0:kW] = x[idx[r], 0:kW] * scale[idx[r]]   (warp per row; scale nullable; idx[r] < 0 gives a zero row)
template <typename T, int kW>
__global__ void __launch_bounds__(kSagWarps * 32)
k_gather_rows(const T* __restrict__ x, int64_t ldx, const int32_t* __restrict__ idx, const float* __restrict__ scale,
              int64_t n_out, T* __restrict__ out, int64_t ldo) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_out; r += n_warps) {
    const int32_t src = idx[r];
    float v[kPer];
    if (src < 0) {                                   // no source row: zeros (the gradient of a dropped edge)
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] = 0.f;
    } else {
      IO::load(x + (size_t)src * ldx, lane, v);
      if (scale) {
        const float s = scale[src];
#pragma unroll
        for (int i = 0; i < kPer; ++i) v[i] *= s;
      }
    }
    IO::store(out + (size_t)r * ldo, lane, v);
  }
}

// ------------------------------------------------------------------ SAGPooling backward (training step)
// Forward: s = tanh(sign * pre), pre_i = sum_{j -> i} w_l . x_j + b + w_r . x_i;  x'_r = x[perm[r]] * s[perm[r]].
// Given dx' [N', kW]:
//   k_sag_bwd_rowdot   ds_r = dx'_r . x[perm[r]];  dpre[perm[r]] = sign * (1 - s^2) * ds_r   (dpre zero elsewhere)
//   k_sag_score<false> t_j = sum_{i: j -> i} dpre_i  over the CSR keyed by SOURCE
//   k_sag_bwd_dx       dx_j = [j kept] s_j dx'_{new_id[j]} + w_l t_j + w_r dpre_j
// and on the host side dw_l = sum_j t_j x_j, dw_r = sum_j dpre_j x_j (bg_sgemm with M = 1), db = sum_j dpre_j (bg_colsum).
template <typename T, int kW>
__global__ void __launch_bounds__(kSagWarps * 32)
k_sag_bwd_rowdot(const T* __restrict__ dxp, const T* __restrict__ x, const int32_t* __restrict__ perm,
                 const float* __restrict__ score, float sign, int64_t n_out, float* __restrict__ dpre) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_out; r += n_warps) {
    const int32_t j = perm[r];
    float a[kPer], b[kPer];
    IO::load(dxp + (size_t)r * kW, lane, a);
    IO::load(x + (size_t)j * kW, lane, b);
    float d = 0.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) d = fmaf(a[i], b[i], d);
    d = warp_sum(d);
    if (lane == 0) {
      const float sj = score[j];
      dpre[j] = sign * (1.f - sj * sj) * d;
    }
  }
}

template <typename T, int kW>
__global__ void __launch_bounds__(kSagWarps * 32)
k_sag_bwd_dx(const T* __restrict__ dxp, const int32_t* __restrict__ new_id, const float* __restrict__ score,
             const float* __restrict__ t, const float* __restrict__ dpre, const float* __restrict__ w_l,
             const float* __restrict__ w_r, int64_t N, T* __restrict__ dx) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  float wl[kPer], wr[kPer];
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int c = IO::col_of(lane, i);
    wl[i] = w_l[c];
    wr[i] = w_r[c];
  }
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < N; j += n_warps) {
    const int32_t nid = new_id[j];
    float v[kPer];
    if (nid >= 0) {
      IO::load(dxp + (size_t)nid * kW, lane, v);
      const float sj = score[j];
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] *= sj;
    } else {
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] = 0.f;
    }
    const float tj = t[j], dj = dpre[j];
#pragma unroll
    for (int i = 0; i < kPer; ++i) v[i] = fmaf(wl[i], tj, fmaf(wr[i], dj, v[i]));
    IO::store(dx + (size_t)j * kW, lane, v);
  }
}

__global__ void k_index_invert(const int32_t* __restrict__ perm, int64_t n, int32_t* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[perm[i]] = (int32_t)i;
}
__global__ void k_index_gather(const int32_t* __restrict__ table, const int32_t* __restrict__ idx, int64_t n,
                               int32_t* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = table[idx[i]];
}

struct SagWorkspace {
  float* p; float* q; int32_t* tile_ptr; int32_t* block_sums;
  int32_t n_edge_blocks; size_t bytes;
};
static inline SagWorkspace sag_workspace_layout(void* base, int64_t N, int64_t E, int64_t G) {
  SagWorkspace w;
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  char* b = static_cast<char*>(base);
  size_t off = 0;
  w.p = reinterpret_cast<float*>(b + off); off += up(sizeof(float) * (size_t)(N > 0 ? N : 1));
  w.q = reinterpret_cast<float*>(b + off); off += up(sizeof(float) * (size_t)(N > 0 ? N : 1));
  w.n_edge_blocks = (int32_t)ceil_div64(E > 0 ? E : 1, kEdgeItemsPerBlock);
  w.block_sums = reinterpret_cast<int32_t*>(b + off); off += up(sizeof(int32_t) * (size_t)w.n_edge_blocks);
  w.tile_ptr = reinterpret_cast<int32_t*>(b + off); off += up(sizeof(int32_t) * (size_t)(G + 1));   // last: the only G-dependent part
  w.bytes = off;
  return w;
}

}  // namespace bg
