// Training-step kernels: what `loss.backward()` and train-mode BatchNorm / Dropout need around
// the forward kernels (reference: TRAIN_FINAL.py:289-297 drives Models/BuckGNN.py:445-458 in
// train mode; autograd of PyG SAGEConv, F.normalize, BatchNorm1d, ReLU, Dropout, global_mean_pool
// and the encoder / decoder MLPs).
//
// One GraphSAGE layer, forward (train):   agg = A x;  z = agg Wl^T + b + x Wr^T;  u = z / |z|   (K2 + K3, u and
//   1/|z| saved);  batch statistics of u (k_col_stats + k_bn_fwd_finalize);  y = drop(relu(a u + shift) + x_prev)
//   (k_bn_act_fwd; a = gamma * invstd, shift = beta - mean * a).
// Backward, given dy:   g = drop'(dy);  dv = g [a u + shift > 0];  column sums S1 = sum dv, S2 = sum dv u
//   (k_col_stats) -> dbeta = S1, dgamma = invstd (S2 - mean S1), and the BatchNorm input gradient
//   du = a dv - k0 - k1 u;  dz = (du - u (u . du)) / |z|  (k_sage_bwd_rows);  then on the tensor cores
//   dagg = dz Wl, dx = dz Wr + A^T dagg (+ g for skip layers), dWl = dz^T agg, dWr = dz^T x  (bg_gemm512 on
//   transposed / chunked operands, k_transpose_chunks + k_reduce_partials for the split-K over nodes).
//
// The row kernels are templates on the row width kW: 512, or 128 for a hidden_channels = 128 model (the `bg_*128` entry
// points; its weight gradients run on bg_wgrad128, gemm128.cuh).
//
// All reductions are two-stage with a fixed order (no floating-point atomics): a training step is
// bit-reproducible for a given seed.
#pragma once
#include "aggregate.cuh"
#include "common.cuh"

namespace bg {

constexpr int kStatWarps = 8;

BG_DEVINL uint32_t hash32(uint32_t h) {
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
// Dropout keep-decision of element (row, col) of a layer: counter-based (stateless), so the backward
// pass regenerates the mask instead of storing it.  thr = p * 2^32; keep iff hash >= thr.
BG_DEVINL bool dropout_keep(uint64_t seed, int64_t row, int col, uint32_t thr) {
  const uint64_t idx = (uint64_t)row * kHidden + (uint64_t)col;
  const uint32_t h = hash32(hash32((uint32_t)idx + (uint32_t)seed) ^ ((uint32_t)(idx >> 32) + (uint32_t)(seed >> 32)));
  return h >= thr;
}
static inline uint32_t dropout_threshold(float p) {
  if (!(p > 0.f)) return 0u;
  const double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
}

template <typename T> BG_DEVINL void row_load(const T* row, int lane, float (&v)[16]) {
  RowFrag<T> f;
  f.load(row, lane);
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = 0.f;
  f.template accumulate<BG_AGGR_SUM>(v);
}
// One row of kW columns per warp: 512 -> RowFrag (16 columns a lane, interleaved), 128 -> 4 consecutive columns a
// lane (one 16-byte / 8-byte access).  The kernels below are templates on kW; their 512 instances are the kernels the
// 512-wide step has always run.
template <typename T, int kW> struct RowIO;
template <typename T> struct RowIO<T, kHidden> {
  static constexpr int kPer = 16;
  static BG_DEVINL int col_of(int lane, int i) { return RowFrag<T>::col_of(lane, i); }
  static BG_DEVINL void load(const T* row, int lane, float (&v)[16]) { row_load<T>(row, lane, v); }
  static BG_DEVINL void store(T* row, int lane, const float (&v)[16]) { RowFrag<T>::store(row, lane, v); }
};
template <typename T> struct RowIO<T, 128> {
  static constexpr int kPer = 4;
  static BG_DEVINL int col_of(int lane, int i) { return 4 * lane + i; }
  static BG_DEVINL void load(const T* row, int lane, float (&v)[4]) {
    if constexpr (sizeof(T) == 4) {
      const float4 q = *reinterpret_cast<const float4*>(row + 4 * lane);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(row + 4 * lane);
      v[0] = Pack16<T>::lo(u.x); v[1] = Pack16<T>::hi(u.x); v[2] = Pack16<T>::lo(u.y); v[3] = Pack16<T>::hi(u.y);
    }
  }
  static BG_DEVINL void store(T* row, int lane, const float (&v)[4]) {
    if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(row + 4 * lane) = make_float4(v[0], v[1], v[2], v[3]);
    else *reinterpret_cast<uint2*>(row + 4 * lane) = make_uint2(Pack16<T>::pack(v[0], v[1]), Pack16<T>::pack(v[2], v[3]));
  }
};

template <typename T, int kW = kHidden>
BG_DEVINL void lane_vec(const float* __restrict__ vec, int lane, float (&v)[RowIO<T, kW>::kPer]) {
#pragma unroll
  for (int i = 0; i < RowIO<T, kW>::kPer; ++i) v[i] = vec[RowIO<T, kW>::col_of(lane, i)];
}
BG_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct DropArgs { uint64_t seed; uint32_t thr; float inv_keep; };

// g = dropout'(dy + dy2) for this lane's columns of row r (the dropout element index stays r * 512 + c at every width)
template <typename T, int kW = kHidden>
BG_DEVINL void load_upstream(const T* __restrict__ dy, const T* __restrict__ dy2, int64_t r, int lane, const DropArgs& d,
                             float (&g)[RowIO<T, kW>::kPer]) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  IO::load(dy + (size_t)r * kW, lane, g);
  if (dy2) {
    float t[kPer];
    IO::load(dy2 + (size_t)r * kW, lane, t);
#pragma unroll
    for (int i = 0; i < kPer; ++i) g[i] += t[i];
  }
  if (d.thr) {
#pragma unroll
    for (int i = 0; i < kPer; ++i)
      g[i] = dropout_keep(d.seed, r, IO::col_of(lane, i), d.thr) ? g[i] * d.inv_keep : 0.f;
  }
}

// ------------------------------------------------------------------ column statistics
// kMode 0: S1 = sum_r u, S2 = sum_r u^2                         (train-mode BatchNorm forward)
// kMode 1: dv = g [a u + shift > 0]; S1 = sum dv, S2 = sum dv u  (BatchNorm backward)
// partial [gridDim.x][2][kW] f32; each CTA owns a contiguous chunk of rows
template <typename T, int kMode, int kW = kHidden>
__global__ void __launch_bounds__(kStatWarps * 32)
k_col_stats(const T* __restrict__ u, const T* __restrict__ dy, const T* __restrict__ dy2, int64_t N,
            const float* __restrict__ a, const float* __restrict__ shift, const DropArgs drop,
            float* __restrict__ partial) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  __shared__ float red[kStatWarps][2][kW];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t chunk = (N + gridDim.x - 1) / gridDim.x;
  const int64_t r_beg = (int64_t)blockIdx.x * chunk, r_end = min(N, r_beg + chunk);
  float s1[kPer], s2[kPer];
  [[maybe_unused]] float av[kPer], sv[kPer];
#pragma unroll
  for (int i = 0; i < kPer; ++i) s1[i] = s2[i] = 0.f;
  if constexpr (kMode == 1) { lane_vec<T, kW>(a, lane, av); lane_vec<T, kW>(shift, lane, sv); }
  for (int64_t r = r_beg + warp; r < r_end; r += kStatWarps) {
    float uv[kPer];
    IO::load(u + (size_t)r * kW, lane, uv);
    if constexpr (kMode == 0) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) { s1[i] += uv[i]; s2[i] = fmaf(uv[i], uv[i], s2[i]); }
    } else {
      float g[kPer];
      load_upstream<T, kW>(dy, dy2, r, lane, drop, g);
#pragma unroll
      for (int i = 0; i < kPer; ++i) {
        const float dv = fmaf(av[i], uv[i], sv[i]) > 0.f ? g[i] : 0.f;
        s1[i] += dv; s2[i] = fmaf(dv, uv[i], s2[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int c = IO::col_of(lane, i);
    red[warp][0][c] = s1[i]; red[warp][1][c] = s2[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * kW; c += blockDim.x) {
    const int k = c / kW, cc = c % kW;
    float v = red[0][k][cc];
#pragma unroll
    for (int w = 1; w < kStatWarps; ++w) v += red[w][k][cc];
    partial[(size_t)blockIdx.x * 2 * kW + c] = v;
  }
}

struct BnVectors {          // [kW] f32 each, device
  float* a;                 // gamma * invstd          (1 without BatchNorm)
  float* shift;             // beta - mean * a         (0 without BatchNorm)
  float* mean;
  float* invstd;
};

// Finalize kernels: kFinalizeCtas (kW / 64) CTAs x 512 threads.  CTA b owns columns [64 b, 64 b + 64); thread (g, cl) sums the
// partial slots p = g, g + 8, ... of column 64 b + cl in fp64 (four interleaved chains), the eight groups are added in
// a fixed order through shared memory, and the threads of group 0 finish their column.  (Round 1 ran ONE CTA of 512
// threads, each walking all ~300 slots of its column: 34 us per launch, 12 launches per training step -- the
// dependent L2 round trips, not the arithmetic, were the cost.)
constexpr int kFinalizeCtas = kHidden / 64;
template <int kW = kHidden>
BG_DEVINL bool sum_partials(const float* __restrict__ partial, int n_parts, int& c, double& s1, double& s2) {
  __shared__ double sh1[8][64], sh2[8][64];
  const int cl = threadIdx.x & 63, g = threadIdx.x >> 6;
  c = blockIdx.x * 64 + cl;
  double a1[4], a2[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) a1[k] = a2[k] = 0.0;
  int p = g;
  for (; p + 24 < n_parts; p += 32) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      a1[k] += (double)partial[(size_t)(p + 8 * k) * 2 * kW + c];
      a2[k] += (double)partial[(size_t)(p + 8 * k) * 2 * kW + kW + c];
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (p + 8 * k < n_parts) {
      a1[k] += (double)partial[(size_t)(p + 8 * k) * 2 * kW + c];
      a2[k] += (double)partial[(size_t)(p + 8 * k) * 2 * kW + kW + c];
    }
  }
  sh1[g][cl] = (a1[0] + a1[1]) + (a1[2] + a1[3]);
  sh2[g][cl] = (a2[0] + a2[1]) + (a2[2] + a2[3]);
  __syncthreads();
  if (g != 0) return false;
  s1 = ((sh1[0][cl] + sh1[1][cl]) + (sh1[2][cl] + sh1[3][cl])) + ((sh1[4][cl] + sh1[5][cl]) + (sh1[6][cl] + sh1[7][cl]));
  s2 = ((sh2[0][cl] + sh2[1][cl]) + (sh2[2][cl] + sh2[3][cl])) + ((sh2[4][cl] + sh2[5][cl]) + (sh2[6][cl] + sh2[7][cl]));
  return true;
}

// Batch mean / biased variance -> a, shift, mean, invstd; running statistics updated as torch.nn.BatchNorm1d does in
// train mode (momentum, unbiased variance) -- Models/BuckGNN.py:163,451.
template <int kW = kHidden>
__global__ void __launch_bounds__(kHidden)
k_bn_fwd_finalize(const float* __restrict__ partial, int n_parts, int64_t N, const float* __restrict__ gamma,
                  const float* __restrict__ beta, float eps, float momentum, float* __restrict__ running_mean,
                  float* __restrict__ running_var, long long* __restrict__ num_batches_tracked, BnVectors out) {
  int c;
  double s1, s2;
  if (!sum_partials<kW>(partial, n_parts, c, s1, s2)) return;
  const double mean = s1 / (double)N;
  double var = s2 / (double)N - mean * mean;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float av = gamma[c] * invstd;
  out.a[c] = av;
  out.shift[c] = beta[c] - (float)mean * av;
  out.mean[c] = (float)mean;
  out.invstd[c] = invstd;
  if (running_mean) {
    const double unbiased = N > 1 ? var * (double)N / (double)(N - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
  if (num_batches_tracked && c == 0) *num_batches_tracked += 1;
}

// dbeta = S1, dgamma = invstd (S2 - mean S1);  du = a dv - k0 - k1 u  with
// k1 = a invstd dgamma / N,  k0 = a S1 / N - k1 mean
template <int kW = kHidden>
__global__ void __launch_bounds__(kHidden)
k_bn_bwd_finalize(const float* __restrict__ partial, int n_parts, int64_t N, const BnVectors bn,
                  float* __restrict__ dgamma, float* __restrict__ dbeta, int accumulate,
                  float* __restrict__ k0, float* __restrict__ k1) {
  int c;
  double s1, s2;
  if (!sum_partials<kW>(partial, n_parts, c, s1, s2)) return;
  const double mean = bn.mean[c], invstd = bn.invstd[c], av = bn.a[c];
  const double dg = invstd * (s2 - mean * s1);
  if (accumulate) { dgamma[c] += (float)dg; dbeta[c] += (float)s1; }
  else { dgamma[c] = (float)dg; dbeta[c] = (float)s1; }
  const double kk1 = av * invstd * dg / (double)N;
  k1[c] = (float)kk1;
  k0[c] = (float)(av * s1 / (double)N - kk1 * mean);
}

// ------------------------------------------------------------------ y = drop(relu(a u + shift) + x_prev)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_bn_act_fwd(const T* __restrict__ u, const T* __restrict__ x_prev, T* __restrict__ y, int64_t N,
             const float* __restrict__ a, const float* __restrict__ shift, const DropArgs drop) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float av[kPer], sv[kPer];
  lane_vec<T, kW>(a, lane, av); lane_vec<T, kW>(shift, lane, sv);
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    float v[kPer];
    IO::load(u + (size_t)r * kW, lane, v);
#pragma unroll
    for (int i = 0; i < kPer; ++i) v[i] = fmaxf(fmaf(av[i], v[i], sv[i]), 0.f);
    if (x_prev) {
      float t[kPer];
      IO::load(x_prev + (size_t)r * kW, lane, t);
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] += t[i];
    }
    if (drop.thr) {
#pragma unroll
      for (int i = 0; i < kPer; ++i)
        v[i] = dropout_keep(drop.seed, r, IO::col_of(lane, i), drop.thr) ? v[i] * drop.inv_keep : 0.f;
    }
    IO::store(y + (size_t)r * kW, lane, v);
  }
}

// ------------------------------------------------------------------ dz rows
// dv = g [a u + shift > 0];  du = a dv - k0 - k1 u;  dz = inv_norm (du - u (u . du));
// dz_scaled = dz / max(deg, 1) (mean aggregation: the row of A^T dagg's operand);  g_out = g (skip layers)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_sage_bwd_rows(const T* __restrict__ u, const T* __restrict__ dy, const T* __restrict__ dy2, int64_t N,
                const float* __restrict__ inv_norm, const int32_t* __restrict__ rowptr,
                const float* __restrict__ a, const float* __restrict__ shift, const float* __restrict__ k0,
                const float* __restrict__ k1, const DropArgs drop, T* __restrict__ dz, T* __restrict__ dz_scaled,
                T* __restrict__ g_out) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float av[kPer], sv[kPer], k0v[kPer], k1v[kPer];
  lane_vec<T, kW>(a, lane, av); lane_vec<T, kW>(shift, lane, sv);
  lane_vec<T, kW>(k0, lane, k0v); lane_vec<T, kW>(k1, lane, k1v);
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    float uv[kPer], g[kPer];
    IO::load(u + (size_t)r * kW, lane, uv);
    load_upstream<T, kW>(dy, dy2, r, lane, drop, g);
    if (g_out) IO::store(g_out + (size_t)r * kW, lane, g);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const float dv = fmaf(av[i], uv[i], sv[i]) > 0.f ? g[i] : 0.f;
      g[i] = fmaf(av[i], dv, -fmaf(k1v[i], uv[i], k0v[i]));      // du
      dot = fmaf(uv[i], g[i], dot);
    }
    dot = warp_sum(dot);
    const float inr = inv_norm ? inv_norm[r] : 1.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) g[i] = inv_norm ? inr * fmaf(-uv[i], dot, g[i]) : g[i];
    IO::store(dz + (size_t)r * kW, lane, g);
    if (dz_scaled) {
      const float id = 1.f / (float)max(rowptr[r + 1] - rowptr[r], 1);
#pragma unroll
      for (int i = 0; i < kPer; ++i) g[i] *= id;
      IO::store(dz_scaled + (size_t)r * kW, lane, g);
    }
  }
}

// ------------------------------------------------------------------ split-K operand layout
// in [n_rows, n_cols] (ld) -> out [n_chunks][out_rows >= n_cols][chunk_k]:  out[s][c][j] = in[s*chunk_k + j][c], 0 beyond
// n_rows (rows c >= n_cols of a chunk are left untouched: the caller zero-fills them when it pads a narrow matrix
// to the 512 rows the tensor-core GEMM multiplies).
// The node dimension becomes the contiguous (K) dimension the tcgen05 operand tiles want; chunk s of the
// split-K is a [n_cols, chunk_k] K-major matrix.   grid (ceil(n_chunks*chunk_k / 32), n_cols / 32), block (32, 8)
template <typename T>
__global__ void __launch_bounds__(256)
k_transpose_chunks(const T* __restrict__ in, int64_t n_rows, int n_cols, int64_t ld, int64_t chunk_k, int out_rows,
                   T* __restrict__ out) {
  __shared__ T tile[32][33];
  const int64_t j0 = (int64_t)blockIdx.x * 32;       // global node index of the tile
  const int c0 = blockIdx.y * 32;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t r = j0 + threadIdx.y + 8 * k;
    tile[threadIdx.y + 8 * k][threadIdx.x] = (r < n_rows) ? in[(size_t)r * ld + c0 + threadIdx.x] : T(0.f);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c0 + threadIdx.y + 8 * k;
    const int64_t j = j0 + threadIdx.x;              // chunk_k is a multiple of 32: a tile never straddles chunks
    const int64_t s = j / chunk_k, jj = j % chunk_k;
    out[((size_t)s * out_rows + c) * chunk_k + jj] = tile[threadIdx.x][threadIdx.y + 8 * k];
  }
}

// out[i] (+)= sum_s partial[s][i], fixed order
__global__ void k_reduce_partials(const float* __restrict__ partial, int n_chunks, int64_t n, float* __restrict__ out,
                                  int accumulate) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = 0.f;
    for (int s = 0; s < n_chunks; ++s) v += partial[(size_t)s * n + i];
    out[i] = accumulate ? out[i] + v : v;
  }
}

// 128-wide weight gradients (bg_wgrad128): partial [n_chunks][256][128] f32 holds, per node chunk, [dWl^T ; dWr^T]
// (row = input feature of lin_l / lin_r, column = output feature).  dW{l,r}[o, i] (+)= sum_s partial[s][{0,128} + i][o],
// summed in chunk order.  Reads are coalesced along o; the 2 x 16 K scattered writes are small next to them.
__global__ void __launch_bounds__(256)
k_reduce_wgrad128(const float* __restrict__ partial, int n_chunks, float* __restrict__ dwl, float* __restrict__ dwr,
                  int accumulate) {
  const int64_t n = 2 * 128 * 128, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const int which = (int)(t >> 14), i = (int)(t >> 7) & 127, o = (int)t & 127;
    float v = 0.f;
    for (int s = 0; s < n_chunks; ++s) v += partial[((size_t)s * 256 + which * 128 + i) * 128 + o];
    float* out = (which ? dwr : dwl) + (size_t)o * 128 + i;
    *out = accumulate ? *out + v : v;
  }
}
// bg_wgrad128_ld: the same sum into column slices of wider weights, dw_k[o * ld_k + i] (+)= sum_s partial[s][128 k + i][o];
// dw1 null: the second half of every pair tile is discarded (a single product).
__global__ void __launch_bounds__(256)
k_reduce_wgrad128_ld(const float* __restrict__ partial, int n_chunks, float* __restrict__ dw0, int64_t ld0,
                     float* __restrict__ dw1, int64_t ld1, int accumulate) {
  const int64_t n = (dw1 ? 2 : 1) * 128 * 128, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const int which = (int)(t >> 14), i = (int)(t >> 7) & 127, o = (int)t & 127;
    float v = 0.f;
    for (int s = 0; s < n_chunks; ++s) v += partial[((size_t)s * 256 + which * 128 + i) * 128 + o];
    float* out = which ? dw1 + (size_t)o * ld1 + i : dw0 + (size_t)o * ld0 + i;
    *out = accumulate ? *out + v : v;
  }
}

// ------------------------------------------------------------------ generic loads by run-time dtype
BG_DEVINL float load_as_float(const void* p, int dtype, size_t i) {
  if (dtype == BG_F32) return static_cast<const float*>(p)[i];
  if (dtype == BG_F16) return __half2float(static_cast<const __half*>(p)[i]);
  return __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]);
}
BG_DEVINL void store_from_float(void* p, int dtype, size_t i, float v) {
  if (dtype == BG_F32) static_cast<float*>(p)[i] = v;
  else if (dtype == BG_F16) static_cast<__half*>(p)[i] = __float2half_rn(v);
  else static_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
}

// column sums of a [rows, cols] matrix: stage 1, grid (ceil(cols/32), n_chunks), block (32, 8) -> partial [n_chunks][cols]
__global__ void __launch_bounds__(256)
k_colsum_partial(const void* __restrict__ in, int dtype, int64_t rows, int cols, int64_t ld, float* __restrict__ partial) {
  __shared__ float red[8][32];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t chunk = (rows + gridDim.y - 1) / gridDim.y;
  const int64_t r_beg = (int64_t)blockIdx.y * chunk, r_end = min(rows, r_beg + chunk);
  float s = 0.f;
  if (c < cols)
    for (int64_t r = r_beg + threadIdx.y; r < r_end; r += 8) s += load_as_float(in, dtype, (size_t)r * ld + c);
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float v = red[0][threadIdx.x];
#pragma unroll
    for (int k = 1; k < 8; ++k) v += red[k][threadIdx.x];
    partial[(size_t)blockIdx.y * cols + c] = v;
  }
}

// ------------------------------------------------------------------ global_mean_pool backward
// dx[r, :] = dpooled[g(r), off:off+512] * w(r);  mean: w = 1/max(cnt,1);  mean_no_super: the graph's last node gets
// 0 and cnt excludes it;  supernode_only: only the last node, w = 1;  supernode_with_pooling (dpooled is [G, 1024] =
// cat[mean_no_super, super]): real nodes take the first half / (cnt - 1), the last node the second half.
// (Models/BuckGNN.py:273-293 in reverse.)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_pool_bwd(const float* __restrict__ dpooled, int64_t ldp, const int32_t* __restrict__ graph_ptr, int G, int mode,
           int64_t N, T* __restrict__ dx) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    int lo = 0, hi = G;                               // last g with graph_ptr[g] <= r
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if ((int64_t)graph_ptr[mid] <= r) lo = mid; else hi = mid; }
    const int64_t beg = graph_ptr[lo], end = graph_ptr[lo + 1];
    const bool last = (r == end - 1);
    float w;
    int64_t off = 0;                                  // column offset into dpooled (the concatenated variant)
    if (mode == BG_POOL_MEAN) w = 1.f / (float)max(end - beg, (int64_t)1);
    else if (mode == BG_POOL_MEAN_NO_SUPER) w = last ? 0.f : 1.f / (float)max(end - beg - 1, (int64_t)1);
    else if (mode == BG_POOL_SUPERNODE_ONLY) w = last ? 1.f : 0.f;
    else { w = last ? 1.f : 1.f / (float)max(end - beg - 1, (int64_t)1); off = last ? kW : 0; }   // cat[mean_no_super, super]
    float v[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) v[i] = w * dpooled[(size_t)lo * ldp + off + IO::col_of(lane, i)];
    IO::store(dx + (size_t)r * kW, lane, v);
  }
}

// ------------------------------------------------------------------ small fp32 GEMM on the CUDA cores
// C[m, n] = sum_k A(m, k) B(k, n) with A(m, k) = a[m*sam + k*sak], B(k, n) = b[k*sbk + n*sbn]; operands of any
// bg_dtype, fp32 math.  For the narrow layers the tensor-core kernel is not shaped for (encoder 16->64->128,
// decoder 512->128->64->out, and their gradients): ~2 % of the step's flops.
// grid (ceil(N/64), ceil(M/64), splits): split z covers k in [z*k_per, (z+1)*k_per) and writes partial z
// ([splits][M][N] f32); k_sgemm_epilogue reduces the splits and applies bias / ReLU / mask.
constexpr int kSgTile = 64, kSgK = 16;
struct SgemmArgs {
  const void* a; const void* b; int a_dtype, b_dtype;
  int64_t sam, sak, sbk, sbn;
  int64_t M, N, K, k_per;
  float* partial;
};

__global__ void __launch_bounds__(256)
k_sgemm(const SgemmArgs p) {
  __shared__ float As[kSgK][kSgTile + 4];
  __shared__ float Bs[kSgK][kSgTile + 4];
  const int t = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * kSgTile, n0 = (int64_t)blockIdx.x * kSgTile;
  const int64_t k_beg = (int64_t)blockIdx.z * p.k_per, k_end = min(p.K, k_beg + p.k_per);
  const int tm = (t / 16) * 4, tn = (t % 16) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool a_kfast = p.sak == 1, b_kfast = p.sbk == 1;
  for (int64_t k0 = k_beg; k0 < k_end; k0 += kSgK) {
#pragma unroll
    for (int e4 = 0; e4 < 4; ++e4) {
      const int e = t + 256 * e4;
      int mm, kk;
      if (a_kfast) { kk = e % kSgK; mm = e / kSgK; } else { mm = e % kSgTile; kk = e / kSgTile; }
      const int64_t m = m0 + mm, k = k0 + kk;
      As[kk][mm] = (m < p.M && k < k_end) ? load_as_float(p.a, p.a_dtype, (size_t)(m * p.sam + k * p.sak)) : 0.f;
      int nn, kb;
      if (b_kfast) { kb = e % kSgK; nn = e / kSgK; } else { nn = e % kSgTile; kb = e / kSgTile; }
      const int64_t n = n0 + nn, k2 = k0 + kb;
      Bs[kb][nn] = (n < p.N && k2 < k_end) ? load_as_float(p.b, p.b_dtype, (size_t)(k2 * p.sbk + n * p.sbn)) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kSgK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][tm]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tn]);
      const float aa[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* dst = p.partial + (size_t)blockIdx.z * p.M * p.N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + tm + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t n = n0 + tn + j;
      if (n < p.N) dst[(size_t)m * p.N + n] = acc[i][j];
    }
  }
}

struct SgemmEpilogue {
  const float* partial; int splits; int64_t M, N;
  const float* bias;              // [N] or null
  int relu;
  const void* mask; int mask_dtype; int64_t mask_ld;   // out *= [mask[m, n] > 0]   (ReLU backward), or null
  void* out; int out_dtype; int64_t ldo; int accumulate;
};

__global__ void k_sgemm_epilogue(const SgemmEpilogue p) {
  const int64_t total = p.M * p.N, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t m = i / p.N, n = i % p.N;
    float v = 0.f;
    for (int s = 0; s < p.splits; ++s) v += p.partial[(size_t)s * total + i];
    if (p.bias) v += p.bias[n];
    if (p.relu) v = fmaxf(v, 0.f);
    if (p.mask && !(load_as_float(p.mask, p.mask_dtype, (size_t)(m * p.mask_ld + n)) > 0.f)) v = 0.f;
    const size_t o = (size_t)(m * p.ldo + n);
    if (p.accumulate) v += load_as_float(p.out, p.out_dtype, o);
    store_from_float(p.out, p.out_dtype, o, v);
  }
}

// ------------------------------------------------------------------ elementwise pieces of the EA-GNN training step
// (Models/BuckGNN.py:375-387 wrapper and GraphNetBlock :552-566 in train mode)
// (templates on the row width kW like the SAGE row kernels above: 128 for a hidden_channels = 128 model, bg_*128)
// y = dropout(x + x_prev)   -- the wrapper's skip + Dropout on node and edge tensors (no activation in between)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_dropout_residual(const T* __restrict__ x, const T* __restrict__ x_prev, T* __restrict__ y, int64_t N, const DropArgs drop) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    float v[kPer];
    IO::load(x + (size_t)r * kW, lane, v);
    if (x_prev) {
      float t[kPer];
      IO::load(x_prev + (size_t)r * kW, lane, t);
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] += t[i];
    }
    if (drop.thr) {
#pragma unroll
      for (int i = 0; i < kPer; ++i)
        v[i] = dropout_keep(drop.seed, r, IO::col_of(lane, i), drop.thr) ? v[i] * drop.inv_keep : 0.f;
    }
    IO::store(y + (size_t)r * kW, lane, v);
  }
}
// out = dropout'(dy + dy2) [act > 0]   (either part optional: thr = 0 -> no dropout, act = null -> no ReLU mask)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_grad_mask(const T* __restrict__ dy, const T* __restrict__ dy2, const T* __restrict__ act, T* __restrict__ out, int64_t N,
            const DropArgs drop) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += n_warps) {
    float g[kPer];
    load_upstream<T, kW>(dy, dy2, r, lane, drop, g);
    if (act) {
      float a[kPer];
      IO::load(act + (size_t)r * kW, lane, a);
#pragma unroll
      for (int i = 0; i < kPer; ++i) g[i] = a[i] > 0.f ? g[i] : 0.f;
    }
    IO::store(out + (size_t)r * kW, lane, g);
  }
}
// scatter_mean backward: every CSR slot of row r receives src[r] / max(count_r, 1)  (count = 1 without `mean`)
template <typename T, int kW = kHidden>
__global__ void __launch_bounds__(256)
k_segment_expand(const T* __restrict__ src, const int32_t* __restrict__ rowptr, int64_t n_rows, int mean, T* __restrict__ out) {
  using IO = RowIO<T, kW>;
  constexpr int kPer = IO::kPer;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows; r += n_warps) {
    const int32_t b = rowptr[r], e = rowptr[r + 1];
    if (e == b) continue;
    float v[kPer];
    IO::load(src + (size_t)r * kW, lane, v);
    if (mean) {
      const float w = 1.f / (float)(e - b);
#pragma unroll
      for (int i = 0; i < kPer; ++i) v[i] *= w;
    }
    for (int32_t s = b; s < e; ++s) IO::store(out + (size_t)s * kW, lane, v);
  }
}

// ------------------------------------------------------------------ device-side collate
// PyG's DataLoader collate (Batch.from_data_list) for a dataset that lives in HBM in concatenated form:
//   store: x_all [sum n, F], ei_all [2, sum e] (node ids LOCAL to their graph), ea_all [sum e, Fe], y_all [G_all],
//          node_ptr / edge_ptr [G_all + 1] (int64)
//   batch of graphs sel[0..G): out x / edge_index (+ node offset of the graph's slot) / edge_attr / batch / y / ptr.
// k_collate_ptr: exclusive scans of the selected graphs' sizes (one CTA; G is at most a few thousand).
__global__ void __launch_bounds__(1024)
k_collate_ptr(const int64_t* __restrict__ sel, int64_t G, const int64_t* __restrict__ node_ptr,
              const int64_t* __restrict__ edge_ptr, int64_t* __restrict__ out_node_ptr, int64_t* __restrict__ out_edge_ptr) {
  __shared__ int64_t carry[2];
  __shared__ int64_t buf[2][1024];
  if (threadIdx.x == 0) { carry[0] = carry[1] = 0; out_node_ptr[0] = 0; out_edge_ptr[0] = 0; }
  __syncthreads();
  for (int64_t base = 0; base < G; base += 1024) {
    const int64_t i = base + threadIdx.x;
    int64_t n = 0, e = 0;
    if (i < G) { const int64_t g = sel[i]; n = node_ptr[g + 1] - node_ptr[g]; e = edge_ptr[g + 1] - edge_ptr[g]; }
    buf[0][threadIdx.x] = n; buf[1][threadIdx.x] = e;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {                 // Hillis-Steele inclusive scan
      int64_t a = 0, b = 0;
      if ((int)threadIdx.x >= off) { a = buf[0][threadIdx.x - off]; b = buf[1][threadIdx.x - off]; }
      __syncthreads();
      buf[0][threadIdx.x] += a; buf[1][threadIdx.x] += b;
      __syncthreads();
    }
    if (i < G) { out_node_ptr[i + 1] = carry[0] + buf[0][threadIdx.x]; out_edge_ptr[i + 1] = carry[1] + buf[1][threadIdx.x]; }
    __syncthreads();
    if (threadIdx.x == 1023) { carry[0] += buf[0][1023]; carry[1] += buf[1][1023]; }
    __syncthreads();
  }
}

BG_DEVINL int64_t slot_of(const int64_t* __restrict__ ptr, int64_t G, int64_t i) {   // last g with ptr[g] <= i
  int64_t lo = 0, hi = G;
  while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (ptr[mid] <= i) lo = mid; else hi = mid; }
  return lo;
}

// one thread per (row, float) of x / edge_attr; rows carry their slot's bookkeeping
__global__ void k_collate_nodes(const float* __restrict__ x_all, int F, const int64_t* __restrict__ sel, int64_t G,
                                const int64_t* __restrict__ node_ptr, const int64_t* __restrict__ out_node_ptr,
                                float* __restrict__ x, int64_t* __restrict__ batch) {
  const int64_t n_out = out_node_ptr[G];
  const int64_t total = n_out * F, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int64_t i = t / F; const int k = (int)(t % F);
    const int64_t g = slot_of(out_node_ptr, G, i);
    const int64_t src = node_ptr[sel[g]] + (i - out_node_ptr[g]);
    x[t] = x_all[src * F + k];
    if (k == 0) batch[i] = g;
  }
}

__global__ void k_collate_edges(const int64_t* __restrict__ ei_all, int64_t E_all, const float* __restrict__ ea_all, int Fe,
                                const int64_t* __restrict__ sel, int64_t G, const int64_t* __restrict__ edge_ptr,
                                const int64_t* __restrict__ out_node_ptr, const int64_t* __restrict__ out_edge_ptr,
                                int64_t* __restrict__ ei, float* __restrict__ ea) {
  const int64_t e_out = out_edge_ptr[G];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < e_out; e += stride) {
    const int64_t g = slot_of(out_edge_ptr, G, e);
    const int64_t src = edge_ptr[sel[g]] + (e - out_edge_ptr[g]);
    const int64_t off = out_node_ptr[g];
    ei[e] = ei_all[src] + off;
    ei[e_out + e] = ei_all[E_all + src] + off;
    for (int k = 0; k < Fe; ++k) ea[e * Fe + k] = ea_all[src * Fe + k];
  }
}

__global__ void k_collate_y(const float* __restrict__ y_all, const int64_t* __restrict__ sel, int64_t G, float* __restrict__ y) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < G) y[i] = y_all[sel[i]];
}

// ------------------------------------------------------------------ loss + metric epilogue (one CTA)
// What TRAIN_FINAL.py:262-263 / :340-341 compute per batch with three host syncs and two scaler uploads:
//   pd = pred * scale + center, td = y * scale + center          (Normalizer.denormalize_eigenvalue, :207-215)
//   loss = mean(|pd - td| / (|td| + eps))                         (RelativeErrorLoss, Utils/Losses.py:755-761)
//   mape = 100 * mean(|td - pd| / |td|)                           (MAPE_error, Dataset_Preparation/Metrics.py:4-12)
//   dpred = d loss / d pred = sign(pd - td) * scale / ((|td| + eps) * G)
// out[0] = loss, out[1] = mape; accum (nullable) [3] += {loss, mape, 1} so an epoch's running sums stay on the device.
__global__ void __launch_bounds__(256)
k_eigen_loss(const float* __restrict__ pred, const float* __restrict__ y, int64_t G, float scale, float center, float eps,
             float* __restrict__ out, float* __restrict__ dpred, float* __restrict__ accum) {
  __shared__ float red[2][256];
  float l = 0.f, m = 0.f;
  for (int64_t i = threadIdx.x; i < G; i += 256) {
    const float pd = fmaf(pred[i], scale, center), td = fmaf(y[i], scale, center);
    const float diff = pd - td, at = fabsf(td);
    l += fabsf(diff) / (at + eps);
    m += fabsf(diff) / at;
    if (dpred) dpred[i] = (diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f)) * scale / ((at + eps) * (float)G);
  }
  red[0][threadIdx.x] = l; red[1][threadIdx.x] = m;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) { red[0][threadIdx.x] += red[0][threadIdx.x + s]; red[1][threadIdx.x] += red[1][threadIdx.x + s]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float loss = red[0][0] / (float)G, mape = 100.f * red[1][0] / (float)G;
    out[0] = loss; out[1] = mape;
    if (accum) { accum[0] += loss; accum[1] += mape; accum[2] += 1.f; }
  }
}

// out[m, n] (f32, ld = n_cols) = in[m, n] * [mask[m, n] > 0]   -- ReLU backward while narrowing a padded GEMM output
__global__ void k_mask_narrow(const void* __restrict__ in, int in_dtype, int64_t ld_in, const void* __restrict__ mask,
                              int mask_dtype, int64_t ld_mask, int64_t M, int n_cols, float* __restrict__ out) {
  const int64_t total = M * n_cols, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t m = i / n_cols; const int n = (int)(i % n_cols);
    const float v = load_as_float(in, in_dtype, (size_t)(m * ld_in + n));
    out[i] = (!mask || load_as_float(mask, mask_dtype, (size_t)(m * ld_mask + n)) > 0.f) ? v : 0.f;
  }
}

// materialise the dropout keep mask of a layer (test hook: lets the oracle apply the same mask)
__global__ void k_dropout_mask(uint64_t seed, uint32_t thr, int64_t n_rows, uint8_t* __restrict__ keep) {
  const int64_t total = n_rows * kHidden, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride)
    keep[i] = dropout_keep(seed, i / kHidden, (int)(i % kHidden), thr) ? 1 : 0;
}

}  // namespace bg
