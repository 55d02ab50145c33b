// K4: segmented global mean pool + regression head.
//
// Replaces `global_mean_pool(x, batch)` and `decoder(pooled).squeeze()` of the
// reference (Models/BuckGNN.py:274, 515-516; decoder shapes :94-100).  HBM bound:
// one read pass over x [N,512].
//   k_pool_partial : grid (G, kPoolSlices); each CTA sums a contiguous slice of one
//                    graph's rows (warp per row subset, fp32), writes partial[g][s][512]
//   k_pool_head    : one CTA per graph: adds the slices in order, divides by
//                    max(count,1), runs Linear(512,128) ReLU Linear(128,64) ReLU
//                    Linear(64,out_dim) in fp32.
// Deterministic: no atomics, fixed reduction order.
#pragma once
#include "common.cuh"
#include "aggregate.cuh"

namespace bg {

constexpr int kPoolSlices = 8;
constexpr int kPoolWarps = 8;

// pooling variants of the reference's get_pooling_layer (Models/BuckGNN.py:246-307); the
// super node is the LAST node of each graph (:252, :256-266)
enum : int { kPoolMean = BG_POOL_MEAN, kPoolMeanNoSuper = BG_POOL_MEAN_NO_SUPER,
             kPoolSuperOnly = BG_POOL_SUPERNODE_ONLY, kPoolSuperWithPooling = BG_POOL_SUPERNODE_WITH_POOLING };

template <typename T, int kW>
__global__ void __launch_bounds__(kPoolWarps * 32)
k_pool_partial(const T* __restrict__ x, const int32_t* __restrict__ graph_ptr, float* __restrict__ partial,
               int exclude_last) {
  __shared__ float red[kPoolWarps][kW];
  const int g = blockIdx.x, slice = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int32_t beg = graph_ptr[g], cnt = max(graph_ptr[g + 1] - beg - (exclude_last ? 1 : 0), 0);
  const int32_t s_beg = beg + (int32_t)((int64_t)cnt * slice / kPoolSlices);
  const int32_t s_end = beg + (int32_t)((int64_t)cnt * (slice + 1) / kPoolSlices);
  constexpr int kCols = kW / 32;                             // columns per lane
  float acc[kCols];
#pragma unroll
  for (int i = 0; i < kCols; ++i) acc[i] = 0.f;
  int32_t r = s_beg + warp;
  if constexpr (kW == kHidden) {
    for (; r + kPoolWarps < s_end; r += 2 * kPoolWarps) {      // two rows in flight per warp
      RowFrag<T> f0, f1;
      f0.load(x + (size_t)r * kHidden, lane);
      f1.load(x + (size_t)(r + kPoolWarps) * kHidden, lane);
      f0.template accumulate<BG_AGGR_SUM>(acc);
      f1.template accumulate<BG_AGGR_SUM>(acc);
    }
    for (; r < s_end; r += kPoolWarps) {
      RowFrag<T> f;
      f.load(x + (size_t)r * kHidden, lane);
      f.template accumulate<BG_AGGR_SUM>(acc);
    }
#pragma unroll
    for (int i = 0; i < kCols; ++i) red[warp][RowFrag<T>::col_of(lane, i)] = acc[i];
  } else {                                                   // narrow rows: lane owns kCols consecutive columns
    static_assert(kCols == 4, "width 128: 4 columns per lane");
    for (; r < s_end; r += kPoolWarps) {
      const T* row = x + (size_t)r * kW + lane * kCols;
      if constexpr (sizeof(T) == 4) {
        const float4 v = *reinterpret_cast<const float4*>(row);
        acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
      } else {
        const uint2 u = *reinterpret_cast<const uint2*>(row);
        Pack16<T>::add2(acc[0], acc[1], u.x);
        Pack16<T>::add2(acc[2], acc[3], u.y);
      }
    }
#pragma unroll
    for (int i = 0; i < kCols; ++i) red[warp][lane * kCols + i] = acc[i];
  }
  __syncthreads();
  float* out = partial + ((size_t)g * kPoolSlices + slice) * kW;
  for (int c = threadIdx.x; c < kW; c += blockDim.x) {
    float v = red[0][c];
#pragma unroll
    for (int w = 1; w < kPoolWarps; ++w) v += red[w][c];
    out[c] = v;
  }
}

// ---- pooling over the 32-row block sums a pool-fused bg_gemm512 epilogue wrote (gemm_tc.cuh, kPool)
// keep[b] = 1 for every 32-row block that holds the first or the last row of a graph: those blocks are read row by
// row from x (the GEMM stored them), every other block lies wholly inside one graph and contributes its block sum.
__global__ void k_pool_block_flags(const int32_t* __restrict__ graph_ptr, int64_t G, int64_t N, uint8_t* __restrict__ keep) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > G) return;
  const int64_t p = graph_ptr[i];
  if (p < N) keep[p >> 5] = 1;
  if (p > 0) keep[(p - 1) >> 5] = 1;
}

// grid (G, kPoolSlices), kW / 2 threads = 2 columns each; same partial[g][slice][kW] layout as k_pool_partial
template <typename T, int kW>
__global__ void __launch_bounds__(256)
k_pool_partial_blocks(const T* __restrict__ x, const float* __restrict__ block_sums, const uint8_t* __restrict__ keep,
                      const int32_t* __restrict__ graph_ptr, float* __restrict__ partial, int exclude_last) {
  static_assert(sizeof(T) == 2, "block sums come from the 16-bit pool-fused epilogue");
  const int g = blockIdx.x, slice = blockIdx.y, t = threadIdx.x;
  const int32_t beg = graph_ptr[g], cnt = max(graph_ptr[g + 1] - beg - (exclude_last ? 1 : 0), 0);
  const int32_t end = beg + cnt;
  float a0 = 0.f, a1 = 0.f;
  if (cnt > 0) {
    const int32_t b0 = beg >> 5, nb = ((end - 1) >> 5) - b0 + 1;
    const int32_t s_b = b0 + (int32_t)((int64_t)nb * slice / kPoolSlices);
    const int32_t e_b = b0 + (int32_t)((int64_t)nb * (slice + 1) / kPoolSlices);
    for (int32_t b = s_b; b < e_b; ++b) {
      if (!keep[b]) {                                 // no graph starts or ends in this block: all 32 rows are ours
        const float2 v = __ldg(reinterpret_cast<const float2*>(block_sums + (size_t)b * kW) + t);
        a0 += v.x; a1 += v.y;
      } else {
        const int32_t r0 = max(beg, b << 5), r1 = min(end, (b << 5) + 32);
        for (int32_t r = r0; r < r1; ++r) {
          const uint32_t u = *(reinterpret_cast<const uint32_t*>(x + (size_t)r * kW) + t);
          a0 = Pack16<T>::add_lo(u, a0); a1 = Pack16<T>::add_hi(u, a1);
        }
      }
    }
  }
  reinterpret_cast<float2*>(partial + ((size_t)g * kPoolSlices + slice) * kW)[t] = make_float2(a0, a1);
}

template <typename T> BG_DEVINL float load_as_float(const T* p) {
  if constexpr (sizeof(T) == 4) return *p; else return (float)*p;
}

// one CTA per graph: pooled feature (kW or 2 kW wide) -> optional MLPPooling Linear+ReLU
// (Models/BuckGNN.py:568-581) -> decoder Linear(in,128) ReLU Linear(128,64) ReLU Linear(64,out)
// (kW = 128: a model of hidden_channels 128, whose 2-layer decoder Linear(128,64) ReLU Linear(64,out) the caller
// passes embedded in the 3-layer one: w1 = [W1; 0], w2 = [I64 | 0], b2 = 0)
template <typename T, int kW>
__global__ void __launch_bounds__(128)
k_pool_head(const T* __restrict__ x, const float* __restrict__ partial, const int32_t* __restrict__ graph_ptr,
            int mode, const float* __restrict__ pre_w, const float* __restrict__ pre_b,
            const float* __restrict__ w1, const float* __restrict__ b1,
            const float* __restrict__ w2, const float* __restrict__ b2,
            const float* __restrict__ w3, const float* __restrict__ b3, int out_dim,
            float* __restrict__ pred, float* __restrict__ pooled_out, const int32_t* __restrict__ nonfinite) {
  __shared__ float feat[2 * kW];
  __shared__ float tmp[kW];
  __shared__ float h1[128];
  __shared__ float h2[64];
  const int g = blockIdx.x, t = threadIdx.x;
  const int32_t n_g = graph_ptr[g + 1] - graph_ptr[g];
  const bool no_super = (mode == kPoolMeanNoSuper || mode == kPoolSuperWithPooling);
  const int in_dim = (mode == kPoolSuperWithPooling) ? 2 * kW : kW;
  if (mode != kPoolSuperOnly) {
    const float cnt = (float)max(n_g - (no_super ? 1 : 0), 1);
    for (int c = t; c < kW; c += 128) {
      const float* pp = partial + (size_t)g * kPoolSlices * kW + c;
      float v = pp[0];
#pragma unroll
      for (int s = 1; s < kPoolSlices; ++s) v += pp[(size_t)s * kW];
      feat[c] = v / cnt;
    }
  }
  if (mode == kPoolSuperOnly || mode == kPoolSuperWithPooling) {
    const int off = (mode == kPoolSuperOnly) ? 0 : kW;
    const T* srow = x + (size_t)(graph_ptr[g + 1] - 1) * kW;
    for (int c = t; c < kW; c += 128) feat[off + c] = (n_g > 0) ? load_as_float(srow + c) : 0.f;
  }
  __syncthreads();
  if (pre_w) {                                   // pooling_mpl: relu(Linear(512,512)(mean))
    for (int o = t; o < kW; o += 128) {
      const float4* wr = reinterpret_cast<const float4*>(pre_w + (size_t)o * kW);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      for (int k = 0; k < kW / 4; ++k) {
        const float4 w = __ldg(wr + k);
        a0 = fmaf(w.x, feat[4 * k], a0); a1 = fmaf(w.y, feat[4 * k + 1], a1);
        a2 = fmaf(w.z, feat[4 * k + 2], a2); a3 = fmaf(w.w, feat[4 * k + 3], a3);
      }
      tmp[o] = fmaxf((a0 + a1) + (a2 + a3) + pre_b[o], 0.f);
    }
    __syncthreads();
    for (int c = t; c < kW; c += 128) feat[c] = tmp[c];
    __syncthreads();
  }
  if (pooled_out)
    for (int c = t; c < in_dim; c += 128) pooled_out[(size_t)g * in_dim + c] = feat[c];
  {  // in_dim -> 128: one output per thread, 4 independent partial sums
    const float4* wr = reinterpret_cast<const float4*>(w1 + (size_t)t * in_dim);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int k = 0; k < in_dim / 4; ++k) {
      const float4 w = __ldg(wr + k);
      a0 = fmaf(w.x, feat[4 * k], a0); a1 = fmaf(w.y, feat[4 * k + 1], a1);
      a2 = fmaf(w.z, feat[4 * k + 2], a2); a3 = fmaf(w.w, feat[4 * k + 3], a3);
    }
    h1[t] = fmaxf((a0 + a1) + (a2 + a3) + b1[t], 0.f);
  }
  __syncthreads();
  if (t < 64) {
    const float* wr = w2 + (size_t)t * 128;
    float a = 0.f;
    for (int k = 0; k < 128; ++k) a = fmaf(__ldg(wr + k), h1[k], a);
    h2[t] = fmaxf(a + b2[t], 0.f);
  }
  __syncthreads();
  if (t < out_dim) {
    const float* wr = w3 + (size_t)t * 64;
    float a = 0.f;
    for (int k = 0; k < 64; ++k) a = fmaf(__ldg(wr + k), h2[k], a);
    // an upstream kernel met values its 16-bit storage format cannot hold (bg_encoder_front): fail loudly
    const bool poisoned = nonfinite != nullptr && *nonfinite != 0;
    pred[(size_t)g * out_dim + t] = poisoned ? __int_as_float(0x7fc00000) : a + b3[t];
  }
}

}  // namespace bg
