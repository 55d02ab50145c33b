// Node-level decoder of a hidden_channels = 128 model (reference Models/BuckGNN.py:518-524, the h <= 128 decoder
// :41-65):  out[r] = W2 relu(W1 x[r] + b1) + b2  for every row r, x [N,128], W1 [64,128], W2 [out_dim,64], out_dim <= 8.
//
// K = 128 and N = 64 are too thin for a tcgen05 / TMEM pipeline (the same reasoning as the encoder front, DESIGN.md
// section 5 K5), so this is a row-streaming kernel: W1 stays in shared memory for the CTA's lifetime and every row of x
// is read once.  Rows are independent: no workspace, no atomics, the same summation order on every run.
//
// 16-bit rows (fp16 / bf16 storage): mma.sync m16n8k16 with fp32 accumulation.  A warp owns 16 rows: 8 k-steps x
// 8 n-tiles, 32 accumulator registers.  The k order inside the product is free as long as A and B agree, so each lane
// loads its A fragments as four 16-byte vectors per row (64 contiguous bytes per row per warp instruction) and W1 is
// staged in the matching column order.  The hidden layer stays in fp32 registers: bias (the accumulator's initial
// value), ReLU, then the 64 -> out_dim product as per-lane partials summed across the quad by shuffles.
//
// fp32 rows (tf32 / fp32 modes): exact fp32 FMAs on CUDA cores, register-tiled like k_encoder_front: 64-row tiles,
// 16 x 16 threads, each thread 4 rows x 4 hidden columns; partials of the second Linear summed over the 16 column
// threads by shuffles.
#pragma once
#include "common.cuh"

namespace bg {

constexpr int kNhK = 128;          // row width
constexpr int kNhH = 64;           // hidden units
constexpr int kNhMaxOut = 8;
constexpr int kNhWarps = 8;
constexpr int kNhW1Ld = kNhK + 8;  // 16-bit W1 row in smem: +16 bytes keeps the fragment loads conflict-free

template <typename T> struct Mma16;
template <> struct Mma16<__half> {
  static BG_DEVINL void run(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};
template <> struct Mma16<__nv_bfloat16> {
  static BG_DEVINL void run(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};

struct NodeHeadSmem16 {
  uint32_t w1[kNhH][kNhW1Ld / 2];   // pairs of 16-bit values, columns in fragment order (see k_node_head128_mma)
  float b1[kNhH];
  float w2[kNhMaxOut][kNhH];
  float b2[kNhMaxOut];
};

// Lane (g, t) = (lane / 4, lane % 4) of a warp reads row r's columns [(4q + t) * 8, +8) as vector q = 0..3.  Its
// halves 0-3 feed k-step 2q, halves 4-7 k-step 2q + 1; within a k-step, halves {0,1} are the fragment's k = 2t, 2t+1
// and halves {2,3} its k = 2t+8, 2t+9.  fragment_col(c) is the k-step-major position of physical column c (even c).
BG_DEVINL int fragment_col(int c) {
  const int q = c >> 5, t = (c >> 3) & 3, h = c & 7;
  return 16 * (2 * q + (h >> 2)) + 8 * ((h >> 1) & 1) + 2 * t;
}

template <typename T>
__global__ void __launch_bounds__(kNhWarps * 32, 2)
k_node_head128_mma(const T* __restrict__ x, int64_t n_rows, const T* __restrict__ w1, const float* __restrict__ b1,
                   const float* __restrict__ w2, const float* __restrict__ b2, int out_dim, float* __restrict__ out) {
  __shared__ __align__(16) NodeHeadSmem16 s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t* w1u = reinterpret_cast<const uint32_t*>(w1);
  for (int i = tid; i < kNhH * kNhK / 2; i += blockDim.x) {
    const int n = i / (kNhK / 2), c = 2 * (i % (kNhK / 2));
    s.w1[n][fragment_col(c) / 2] = w1u[i];
  }
  if (tid < kNhH) s.b1[tid] = b1[tid];
  for (int i = tid; i < kNhMaxOut * kNhH; i += blockDim.x) s.w2[i / kNhH][i % kNhH] = (i / kNhH) < out_dim ? w2[i] : 0.f;
  if (tid < kNhMaxOut) s.b2[tid] = tid < out_dim ? b2[tid] : 0.f;
  __syncthreads();

  const int g = lane >> 2, t = lane & 3;
  const int64_t n_tiles = (n_rows + 15) / 16;
  for (int64_t tile = (int64_t)blockIdx.x * kNhWarps + warp; tile < n_tiles; tile += (int64_t)gridDim.x * kNhWarps) {
    const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
    uint4 v0[4], v1[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      v0[q] = r0 < n_rows ? ldg_nc_v4(x + r0 * kNhK + (4 * q + t) * 8) : make_uint4(0, 0, 0, 0);
      v1[q] = r1 < n_rows ? ldg_nc_v4(x + r1 * kNhK + (4 * q + t) * 8) : make_uint4(0, 0, 0, 0);
    }
    float c[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float ba = s.b1[8 * j + 2 * t], bb = s.b1[8 * j + 2 * t + 1];
      c[j][0] = ba; c[j][1] = bb; c[j][2] = ba; c[j][3] = bb;
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const int q = ks >> 1;
      uint32_t a[4];
      if (ks & 1) { a[0] = v0[q].z; a[1] = v1[q].z; a[2] = v0[q].w; a[3] = v1[q].w; }
      else        { a[0] = v0[q].x; a[1] = v1[q].x; a[2] = v0[q].y; a[3] = v1[q].y; }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        Mma16<T>::run(c[j], a, s.w1[8 * j + g][8 * ks + t], s.w1[8 * j + g][8 * ks + t + 4]);
    }
    // ReLU, then this lane's share of the second Linear: hidden columns 8j + 2t, 8j + 2t + 1 of rows g and g + 8
    float p0[kNhMaxOut], p1[kNhMaxOut];
#pragma unroll
    for (int o = 0; o < kNhMaxOut; ++o) {
      float s0 = 0.f, s1 = 0.f;
      if (o < out_dim) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 w = *reinterpret_cast<const float2*>(&s.w2[o][8 * j + 2 * t]);
          s0 = fmaf(w.x, fmaxf(c[j][0], 0.f), s0); s0 = fmaf(w.y, fmaxf(c[j][1], 0.f), s0);
          s1 = fmaf(w.x, fmaxf(c[j][2], 0.f), s1); s1 = fmaf(w.y, fmaxf(c[j][3], 0.f), s1);
        }
      }
      p0[o] = s0; p1[o] = s1;
    }
#pragma unroll
    for (int o = 0; o < kNhMaxOut; ++o) {
      if (o < out_dim) {
#pragma unroll
        for (int m = 1; m <= 2; m <<= 1) {
          p0[o] += __shfl_xor_sync(0xffffffffu, p0[o], m);
          p1[o] += __shfl_xor_sync(0xffffffffu, p1[o], m);
        }
      }
    }
    // every lane of the quad now holds both rows' sums; lane t stores outputs t and t + 4
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int o = t + 4 * h;
      float y0 = 0.f, y1 = 0.f;
#pragma unroll
      for (int oo = 0; oo < kNhMaxOut; ++oo)       // selects, not a dynamic index into registers
        if (oo == o) { y0 = p0[oo]; y1 = p1[oo]; }
      if (o < out_dim) {
        if (r0 < n_rows) out[r0 * out_dim + o] = y0 + s.b2[o];
        if (r1 < n_rows) out[r1 * out_dim + o] = y1 + s.b2[o];
      }
    }
  }
}

constexpr int kNhRows32 = 64;      // rows per tile of the fp32 kernel
constexpr int kNhXLd = kNhK + 4;   // fp32 row in smem: a warp's two row groups (rows 4 apart) read disjoint banks

struct NodeHeadSmem32 {
  float w1t[kNhK][kNhH];            // [k][n]
  float xs[kNhRows32][kNhXLd];      // [m][k]
  float b1[kNhH];
  float w2[kNhMaxOut][kNhH];
  float b2[kNhMaxOut];
};

__global__ void __launch_bounds__(256, 2)
k_node_head128_f32(const float* __restrict__ x, int64_t n_rows, const float* __restrict__ w1, const float* __restrict__ b1,
                   const float* __restrict__ w2, const float* __restrict__ b2, int out_dim, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char nh_smem_raw[];
  NodeHeadSmem32& s = *reinterpret_cast<NodeHeadSmem32*>(nh_smem_raw);
  const int tid = threadIdx.x;
  for (int i = tid; i < kNhH * kNhK; i += blockDim.x) s.w1t[i % kNhK][i / kNhK] = w1[i];
  if (tid < kNhH) s.b1[tid] = b1[tid];
  for (int i = tid; i < kNhMaxOut * kNhH; i += blockDim.x) s.w2[i / kNhH][i % kNhH] = (i / kNhH) < out_dim ? w2[i] : 0.f;
  if (tid < kNhMaxOut) s.b2[tid] = tid < out_dim ? b2[tid] : 0.f;

  const int tx = tid & 15, ty = tid >> 4;          // hidden columns 4tx..4tx+3 of rows 4ty..4ty+3
  const int64_t n_tiles = (n_rows + kNhRows32 - 1) / kNhRows32;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m0 = tile * kNhRows32;
    __syncthreads();                               // the previous tile's reads of xs are done (and the weights staged)
    for (int i = tid; i < kNhRows32 * kNhK / 4; i += blockDim.x) {
      const int m = i / (kNhK / 4), k4 = i % (kNhK / 4);
      const uint4 v = m0 + m < n_rows ? ldg_nc_v4(x + (m0 + m) * kNhK + 4 * k4) : make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(&s.xs[m][4 * k4]) = v;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = s.b1[4 * tx + b];
#pragma unroll 2
    for (int k = 0; k < kNhK; k += 4) {
      float xa[4][4], wa[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float4 v = *reinterpret_cast<const float4*>(&s.xs[4 * ty + a][k]);
        xa[a][0] = v.x; xa[a][1] = v.y; xa[a][2] = v.z; xa[a][3] = v.w;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 v = *reinterpret_cast<const float4*>(&s.w1t[k + kk][4 * tx]);
        wa[kk][0] = v.x; wa[kk][1] = v.y; wa[kk][2] = v.z; wa[kk][3] = v.w;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(xa[a][kk], wa[kk][b], acc[a][b]);
    }
    float p[4][kNhMaxOut];
#pragma unroll
    for (int o = 0; o < kNhMaxOut; ++o) {
      const float4 w = *reinterpret_cast<const float4*>(&s.w2[o][4 * tx]);
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        float v = 0.f;
        if (o < out_dim) {
          v = fmaf(w.x, fmaxf(acc[a][0], 0.f), v); v = fmaf(w.y, fmaxf(acc[a][1], 0.f), v);
          v = fmaf(w.z, fmaxf(acc[a][2], 0.f), v); v = fmaf(w.w, fmaxf(acc[a][3], 0.f), v);
        }
        p[a][o] = v;
      }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int o = 0; o < kNhMaxOut; ++o)
        if (o < out_dim)
#pragma unroll
          for (int m = 1; m <= 8; m <<= 1) p[a][o] += __shfl_xor_sync(0xffffffffu, p[a][o], m);
    // the 16 column threads of a row group hold all 4 x 8 sums; thread tx stores entries e = 8a + o with e % 16 == tx
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int o = 0; o < kNhMaxOut; ++o)
        if (((8 * a + o) & 15) == tx && o < out_dim && m0 + 4 * ty + a < n_rows)
          out[(m0 + 4 * ty + a) * out_dim + o] = p[a][o] + s.b2[o];
  }
}

}  // namespace bg
