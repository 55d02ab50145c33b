// Backward of the 'max' neighbourhood aggregation (SAGEConv(aggr='max'), Models/BuckGNN.py:171-176, 459-471) for the
// training step.
//
// Forward: agg_i[c] = max_{j -> i} x_j[c]  (0 for a node without in-edges).  The gradient follows what autograd gives
// the reference when PyG reduces with torch's `scatter_reduce_(..., 'amax', include_self=False)` on a zero-initialised
// output (its path without torch_scatter): the upstream gradient of (i, c) is shared EVENLY by all neighbours that
// attain the maximum, and the zero-initialised output element counts as one more sharer when the maximum is 0 --
//     n_i[c]  = [agg_i[c] == 0] + #{j -> i : x_j[c] == agg_i[c]}
//     dx_j[c] = sum_{i : j -> i} [x_j[c] == agg_i[c]] * dagg_i[c] / n_i[c]
// (after a ReLU ties at 0 are the common case, so this detail matters).  Two gather passes, no atomics:
//   kMode 0 over the CSR keyed by TARGET:  w_i = dagg_i / n_i                       (ref = agg_i, neighbours x_j)
//   kMode 1 over the CSR keyed by SOURCE:  dx_j = sum_i [agg_i == x_j] w_i          (ref = x_j,  neighbours agg_i, w_i)
// Rows up to the big-row threshold: one warp per row.  Hub rows: kMaxBwdSlices CTAs per row, each over a contiguous slice
// of the neighbour list with its warps on interleaved neighbours; partial sums are added in a fixed order.
// Templates on the row width kW (512, or 128 for a hidden_channels = 128 model).
#pragma once
#include "common.cuh"
#include "aggregate.cuh"
#include "train.cuh"

namespace bg {

constexpr int kMaxBwdWarps = 8;          // row kernel: one warp per row
constexpr int kMaxBwdBigWarps = 16;      // hub kernels: warps of a CTA take interleaved neighbours (32 KB of partials)
constexpr int kMaxBwdSlices = 8;         // CTAs per hub row

// acc += [b == ref] * (kMode == 0 ? 1 : w) over neighbours col[beg + first], col[beg + first + step], ...
template <typename T, int kMode, int kW = kHidden>
BG_DEVINL void match_accumulate(const float (&ref)[RowIO<T, kW>::kPer], const T* __restrict__ b, const T* __restrict__ w,
                                const int32_t* __restrict__ col, int32_t beg, int32_t end, int first, int step, int lane,
                                float (&acc)[RowIO<T, kW>::kPer]) {
  constexpr int kPer = RowIO<T, kW>::kPer;
  int32_t e = beg + first;
  if constexpr (kMode == 0) {
    for (; e + 3 * step < end; e += 4 * step) {               // counting pass: four neighbour rows in flight
      float v0[kPer], v1[kPer], v2[kPer], v3[kPer];
      RowIO<T, kW>::load(b + (size_t)col[e] * kW, lane, v0);
      RowIO<T, kW>::load(b + (size_t)col[e + step] * kW, lane, v1);
      RowIO<T, kW>::load(b + (size_t)col[e + 2 * step] * kW, lane, v2);
      RowIO<T, kW>::load(b + (size_t)col[e + 3 * step] * kW, lane, v3);
#pragma unroll
      for (int i = 0; i < kPer; ++i)
        acc[i] += ((v0[i] == ref[i] ? 1.f : 0.f) + (v1[i] == ref[i] ? 1.f : 0.f)) +
                  ((v2[i] == ref[i] ? 1.f : 0.f) + (v3[i] == ref[i] ? 1.f : 0.f));
    }
  }
  for (; e + step < end; e += 2 * step) {                     // two neighbour rows in flight
    const int32_t k0 = col[e], k1 = col[e + step];
    float v0[kPer], v1[kPer];
    RowIO<T, kW>::load(b + (size_t)k0 * kW, lane, v0);
    RowIO<T, kW>::load(b + (size_t)k1 * kW, lane, v1);
    if constexpr (kMode == 0) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) acc[i] += (v0[i] == ref[i] ? 1.f : 0.f) + (v1[i] == ref[i] ? 1.f : 0.f);
    } else {
      float w0[kPer], w1[kPer];
      RowIO<T, kW>::load(w + (size_t)k0 * kW, lane, w0);
      RowIO<T, kW>::load(w + (size_t)k1 * kW, lane, w1);
#pragma unroll
      for (int i = 0; i < kPer; ++i) acc[i] += (v0[i] == ref[i] ? w0[i] : 0.f) + (v1[i] == ref[i] ? w1[i] : 0.f);
    }
  }
  for (; e < end; e += step) {
    const int32_t k0 = col[e];
    float v0[kPer];
    RowIO<T, kW>::load(b + (size_t)k0 * kW, lane, v0);
    if constexpr (kMode == 0) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) acc[i] += (v0[i] == ref[i] ? 1.f : 0.f);
    } else {
      float w0[kPer];
      RowIO<T, kW>::load(w + (size_t)k0 * kW, lane, w0);
#pragma unroll
      for (int i = 0; i < kPer; ++i) acc[i] += (v0[i] == ref[i] ? w0[i] : 0.f);
    }
  }
}

// kMode 0: out_r = d_r / (acc + [ref == 0]);   kMode 1: out_r = acc
template <typename T, int kMode, int kW = kHidden>
BG_DEVINL void match_finish(const float (&ref)[RowIO<T, kW>::kPer], const T* __restrict__ d_row, float (&acc)[RowIO<T, kW>::kPer], int lane) {
  constexpr int kPer = RowIO<T, kW>::kPer;
  if constexpr (kMode == 0) {
    float d[kPer];
    RowIO<T, kW>::load(d_row, lane, d);
#pragma unroll
    for (int i = 0; i < kPer; ++i) acc[i] = d[i] / (acc[i] + (ref[i] == 0.f ? 1.f : 0.f));
  }
}

// (128-wide rows: at least 4 CTAs per SM requested -- without the hint ptxas packs the fp32 instance into 32 registers
//  and spills)
template <typename T, int kMode, int kW = kHidden>
__global__ void __launch_bounds__(kMaxBwdWarps * 32, kW == kHidden ? 0 : 4)
k_max_bwd_rows(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ w, const T* __restrict__ d,
               const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N, T* __restrict__ out) {
  constexpr int kPer = RowIO<T, kW>::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    const int32_t beg = rowptr[r], end = rowptr[r + 1];
    if (end - beg > kBigRowThreshold) continue;                // k_max_bwd_big
    float ref[kPer], acc[kPer];
    RowIO<T, kW>::load(a + (size_t)r * kW, lane, ref);
#pragma unroll
    for (int i = 0; i < kPer; ++i) acc[i] = 0.f;
    match_accumulate<T, kMode, kW>(ref, b, w, col, beg, end, 0, 1, lane, acc);
    match_finish<T, kMode, kW>(ref, d + (size_t)r * kW, acc, lane);
    RowIO<T, kW>::store(out + (size_t)r * kW, lane, acc);
  }
}

// Hub rows: grid (n_big, kMaxBwdSlices).  CTA (b, s) takes the s-th contiguous slice of the row's neighbour list, its
// warps interleaved neighbours of the slice; the CTA's partial sum goes to partial[b][s][kW] and k_max_bwd_big_finish
// adds the slices in order (no atomics).
template <typename T, int kMode, int kW = kHidden>
__global__ void __launch_bounds__(kMaxBwdBigWarps * 32)
k_max_bwd_big(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ w,
              const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ big_rows,
              float* __restrict__ partial) {
  constexpr int kPer = RowIO<T, kW>::kPer;
  __shared__ float red[kMaxBwdBigWarps][kW];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int32_t r = big_rows[blockIdx.x];
  const int32_t row_beg = rowptr[r], deg = rowptr[r + 1] - row_beg;
  const int32_t beg = row_beg + (int32_t)((int64_t)deg * blockIdx.y / kMaxBwdSlices);
  const int32_t end = row_beg + (int32_t)((int64_t)deg * (blockIdx.y + 1) / kMaxBwdSlices);
  float ref[kPer], acc[kPer];
  RowIO<T, kW>::load(a + (size_t)r * kW, lane, ref);
#pragma unroll
  for (int i = 0; i < kPer; ++i) acc[i] = 0.f;
  match_accumulate<T, kMode, kW>(ref, b, w, col, beg, end, warp, kMaxBwdBigWarps, lane, acc);
#pragma unroll
  for (int i = 0; i < kPer; ++i) red[warp][RowIO<T, kW>::col_of(lane, i)] = acc[i];
  __syncthreads();
  float* out = partial + ((size_t)blockIdx.x * kMaxBwdSlices + blockIdx.y) * kW;
  for (int c = threadIdx.x; c < kW; c += blockDim.x) {
    float v = red[0][c];
#pragma unroll
    for (int k = 1; k < kMaxBwdBigWarps; ++k) v += red[k][c];
    out[c] = v;
  }
}

template <typename T, int kMode, int kW = kHidden>
__global__ void __launch_bounds__(32)
k_max_bwd_big_finish(const T* __restrict__ a, const T* __restrict__ d, const int32_t* __restrict__ big_rows,
                     const float* __restrict__ partial, T* __restrict__ out) {
  constexpr int kPer = RowIO<T, kW>::kPer;
  const int lane = threadIdx.x;
  const int32_t r = big_rows[blockIdx.x];
  float ref[kPer], acc[kPer];
  RowIO<T, kW>::load(a + (size_t)r * kW, lane, ref);
  const float* p = partial + (size_t)blockIdx.x * kMaxBwdSlices * kW;
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int c = RowIO<T, kW>::col_of(lane, i);
    float v = p[c];
#pragma unroll
    for (int k = 1; k < kMaxBwdSlices; ++k) v += p[(size_t)k * kW + c];
    acc[i] = v;
  }
  match_finish<T, kMode, kW>(ref, d + (size_t)r * kW, acc, lane);
  RowIO<T, kW>::store(out + (size_t)r * kW, lane, acc);
}

}  // namespace bg
