// K3 at width 128: tcgen05 tile GEMM whose output row is 128 wide, with the SAGE update epilogue fused in.
//
//   out[m, 0:128] = epilogue( sum_s A_s[m, :] . B_s^T )       (up to BG_MAX_GEMM_SEGMENTS K-segments, B_s [128, k_s])
//
// The update GEMM of a hidden_channels = 128 GraphSAGE model (the reference's default width, Models/BuckGNN.py:10)
// and its encoder's last Linear.  A kernel of its own rather than a width parameter of k_gemm512: that one splits the
// 512 columns into two 256-column halves held by two warpgroups that exchange the row's sum of squares; here one
// thread owns a whole 128-column row, so the L2 norm is thread-local.
//
// One persistent CTA pair per SM pair (tcgen05 cta_group::2), 12 warps per CTA:
//   warp 0     TMA producer: this CTA's 128 activation rows x 128 B of K and its 64 of the 128 weight rows into an
//              8-stage ring of 128B-swizzled K-major tiles (24 KB a stage: at K = 256 two tiles of A are in flight)
//   warp 1     allocates 256 TMEM columns = two 128-column accumulators; in the leader CTA one elected lane issues
//              tcgen05.mma (M = 256 over the pair, N = 128) into accumulator (tile iteration & 1)
//   warps 2-3  idle (warpgroup alignment: an epilogue warp may only read the TMEM lane quarter warp % 4)
//   warps 4-11 epilogue, two warpgroups; warpgroup g drains the accumulator of the iterations of parity g, so the
//              next tile's MMAs and epilogue run while a tile is still in its epilogue.  One TMEM lane (= output row)
//              per thread: pass 1 reads the row once for its sum of squares (normalize only), pass 2 re-reads it 128 B
//              of output at a time, applies bias / normalize / BN / ReLU / skip in fp32 (one rounding of the result)
//              and moves the rows through a 4 KB swizzled staging tile per warp, so that global loads and stores are
//              coalesced (8 lanes per 128-byte row piece).
// kGather (bg_gemm128_gathered, the edge GEMMs of a 128-wide EA-GNN layer): up to two rows G_k[gidx_k[m], 0:128] of
// the output dtype are added to output row m before the activation, out = relu(acc + bias + G_0[i0] + G_1[i1]), in fp32
// with one rounding of the result.  They travel like the skip rows (8 lanes per 128-byte row piece, through the staging
// tile), the row index read once per row and broadcast by shuffle.
// kMn (bg_wgrad128, the weight gradients of a 128-wide SAGE layer): both operands MN-major, read in place from row-major
// [n_rows, 128] matrices (no transposed copies), the reduction over nodes.  Tile t = node chunk t: the CTA of rank 0
// loads agg^T, rank 1 loads x^T as its 128 rows of the M = 256 A operand, both CTAs their 64-column half of dz as B, so
// one tile yields [dWl^T ; dWr^T] of the chunk (fp32, plain epilogue) and k_reduce_wgrad128 sums the chunks.
// The kernel streams: at K = 256 (fp16) a CTA pair reads 256 KB of operands per 256 x 128 x 256 MACs, so HBM, not
// the tensor core, bounds it.  No setmaxnreg: every warp keeps the launch allocation (168 registers).
#pragma once
#include "gemm_tc.cuh"

namespace bg {

constexpr int kW128 = 128;                                     // output columns
constexpr int kG128BRows = kW128 / 2;                          // weight rows held by one CTA of the pair
constexpr int kG128BTileBytes = kG128BRows * kStageKBytes;     // 8 KB
constexpr int kG128StageBytes = kATileBytes + kG128BTileBytes; // 24 KB
constexpr int kG128Stages = 8;
constexpr int kG128MiscBytes = 256;                            // mbarriers + TMEM address slot
constexpr int kG128SmemBytes = 1024 + kG128Stages * kG128StageBytes + kEpiWarps * kEpiStageBytes + kG128MiscBytes;
static_assert(kG128SmemBytes <= 232448, "exceeds the 227 KB of dynamic shared memory a CTA may have");
static_assert((2 * kG128Stages + 4) * 8 + 4 <= kG128MiscBytes, "mbarriers overlap the TMEM address slot");

struct alignas(64) Gemm128Params {
  GemmSeg seg[BG_MAX_GEMM_SEGMENTS];
  int32_t kblocks[BG_MAX_GEMM_SEGMENTS];
  int32_t n_seg;
  int32_t k_elems_per_block;        // 64 (16-bit operands) or 32 (tf32)
  uint32_t a_fmt, b_fmt;            // UMMA operand formats: 0 f16, 1 bf16, 2 tf32
  int32_t n_tiles;                  // row tiles of 256 rows (one per CTA pair and iteration)
  int32_t normalize, relu;
  int64_t m;
  void* out;                        // [M, 128] of the output dtype, leading dimension ldo (elements)
  int64_t ldo;
  const void* residual;             // [M, 128] skip rows of the output dtype (ld = ldr), or null
  int64_t ldr;
  float* inv_norm_out;              // [M] f32 or null: 1 / max(|row|, eps) of normalized rows
  float* pool_sums;                 // kPool: [ceil(M/32), 128] f32 column sums of every 32-row block of the output rows
  const uint8_t* pool_keep;         // kPool: [ceil(M/32)] only blocks with a non-zero flag are also stored to `out`
  float bias[kW128];                // epilogue vectors by value -> constant bank
  float scale[kW128];               // 1 when there is no BN
  float shift[kW128];               // 0 when there is no BN
  int64_t chunk_k;                  // kMn: nodes per chunk (a multiple of k_elems_per_block)
  // kGather (appended: the fields above keep their constant-bank offsets)
  const void* gather[2];            // [*, 128] row-major matrices of the output dtype, ld = gather_ld
  const int32_t* gidx[2];           // [M] row index into gather[k]
  int32_t n_gather;                 // 1 or 2
  int64_t gather_ld;
};

// One epilogue warp: 32 TMEM lanes = 32 output rows of the tiles of parity g.  kPool as in k_gemm512 (last layer of a
// graph-level model, 16-bit output): per 32-row block and column the fp32 sum of the stored (rounded) values goes to
// pool_sums, and only the blocks flagged in pool_keep are stored.
template <typename TOut, bool kRes, bool kPool, bool kGather = false>
BG_DEVINL void epilogue128_warp(const Gemm128Params& p, const uint32_t tmem_base, const uint32_t stage_u32,
                                const uint32_t tmem_full_bar, const uint32_t tmem_empty_bar, const uint32_t rank,
                                const int tile0, const int tile_stride, const int g) {
  static_assert(!kPool || (sizeof(TOut) == 2 && !kRes), "pool-fused epilogue: 16-bit output, no skip rows");
  static_assert(!kGather || (!kRes && !kPool), "gathered addends: no skip rows, no pool fusion");
  constexpr bool kOut16 = sizeof(TOut) == 2;
  constexpr size_t esz = sizeof(TOut);
  constexpr int kChunkCols = 128 / (int)esz;                    // output columns per 128-byte row piece: 64 / 32
  constexpr int kChunks = kW128 / kChunkCols;                   // 2 / 4
  constexpr int kPer = 16 / (int)esz;                           // columns per 16-byte piece: 8 / 4
  constexpr int kLoads = kChunkCols / 32;                       // 32-column TMEM loads per chunk
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int q = warp & 3;                                       // TMEM lane quarter this warp may read
  const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * kW128);
  const uint32_t my_row = stage_u32 + (uint32_t)lane * 128u;
  const uint32_t my_sw = (uint32_t)(lane & 7);
  const int r4 = lane >> 3, piece = lane & 7;
  const uint32_t coop_even = stage_u32 + (uint32_t)r4 * 128u + (((uint32_t)piece ^ (uint32_t)r4) << 4);
  const uint32_t coop_odd = stage_u32 + (uint32_t)(4 + r4) * 128u + (((uint32_t)piece ^ (uint32_t)(4 + r4)) << 4);
  const size_t out_row_bytes = (size_t)p.ldo * esz;
  uint32_t j = 0;
  for (int tile = tile0 + g * tile_stride; tile < p.n_tiles; tile += 2 * tile_stride, ++j) {
    const int64_t warp_row0 = (int64_t)tile * (2 * kTileM) + (int64_t)rank * kTileM + q * 32;
    const int64_t m_row = warp_row0 + lane;
    const int rows_here = (int)min((int64_t)32, p.m - warp_row0);                 // <= 0: nothing to store
    [[maybe_unused]] bool keep_rows = true;
    if constexpr (kPool) keep_rows = rows_here > 0 && p.pool_keep[warp_row0 >> 5] != 0;   // warp-uniform
    // skip rows of one 128-byte chunk for the warp's 32 rows: pass t covers rows 4t..4t+3, 8 lanes x 16 B each
    [[maybe_unused]] uint4 pre[kRes ? 8 : 1];
    [[maybe_unused]] const char* res_base = nullptr;
    if constexpr (kRes)
      res_base = reinterpret_cast<const char*>(p.residual) + (size_t)(warp_row0 + r4) * p.ldr * esz + piece * 16;
    // kGather: gathered rows of one 128-byte chunk in the same layout, one matrix at a time (G_1 is loaded only after
    // G_0 has been folded into the accumulator registers: holding both would spill the 16-bit instances)
    [[maybe_unused]] int32_t gi[2] = {0, 0};
    [[maybe_unused]] uint4 gpre[kGather ? 8 : 1];
    if constexpr (kGather) {
      if (m_row < p.m) { gi[0] = p.gidx[0][m_row]; if (p.n_gather > 1) gi[1] = p.gidx[1][m_row]; }
    }
    auto fetch = [&](int ch) {
      if constexpr (kRes) {
#pragma unroll
        for (int t = 0; t < 8; ++t)
          pre[t] = (t * 4 + r4 < rows_here) ? ldg_nc_v4(res_base + (size_t)t * 4 * p.ldr * esz + ch * 128)
                                            : make_uint4(0u, 0u, 0u, 0u);
      }
    };
    [[maybe_unused]] auto fetch_gather = [&](int k, int ch) {
      const char* g_base = reinterpret_cast<const char*>(p.gather[k]) + piece * 16 + ch * 128;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int32_t n = __shfl_sync(0xffffffffu, gi[k], t * 4 + r4);
        gpre[t] = (t * 4 + r4 < rows_here) ? ldg_nc_v4(g_base + (size_t)n * p.gather_ld * esz) : make_uint4(0u, 0u, 0u, 0u);
      }
    };
    // adds the 16-byte piece `u` of a gathered row (kPer values of the output dtype) to v[0..kPer) in fp32
    [[maybe_unused]] auto add_piece = [&](float* v, const uint4 u) {
      const uint32_t au[4] = {u.x, u.y, u.z, u.w};
      if constexpr (kOut16) {
#pragma unroll
        for (int e = 0; e < 4; ++e) Pack16<TOut>::add2(v[2 * e], v[2 * e + 1], au[e]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] += __uint_as_float(au[e]);
      }
    };
    fetch(0);                                                   // in flight while the MMAs run
    if constexpr (kGather) fetch_gather(0, 0);

    mbar_wait(tmem_full_bar, j & 1u, kTagTmemFull);
    tc_fence_after();

    // ---- pass 1 (normalize): the row's sum of squares of acc + bias, four independent chains
    float inv = 1.f;
    if (p.normalize) {
      float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < kW128 / 32; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(taddr + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float v = __uint_as_float(r[e]) + p.bias[c * 32 + e];
          s[e & 3] = fmaf(v, v, s[e & 3]);
        }
      }
      inv = 1.f / fmaxf(sqrtf((s[0] + s[1]) + (s[2] + s[3])), 1e-12f);
      if (p.inv_norm_out != nullptr && m_row < p.m) p.inv_norm_out[m_row] = inv;
    }

    // ---- pass 2: 128-byte output pieces of the row through the warp's staging tile
    char* out_base = reinterpret_cast<char*>(p.out) + (size_t)(warp_row0 + r4) * out_row_bytes + piece * 16;
#pragma unroll
    for (int ch = 0; ch < kChunks; ++ch) {
      if constexpr (kRes) {                                     // stage the skip rows, then prefetch the next chunk's
#pragma unroll
        for (int t = 0; t < 8; ++t) sts_v4(((t & 1) ? coop_odd : coop_even) + (uint32_t)(t >> 1) * 1024u, pre[t]);
        __syncwarp();
        if (ch + 1 < kChunks) fetch(ch + 1);
      }
      uint32_t r[kChunkCols];
#pragma unroll
      for (int l = 0; l < kLoads; ++l) tmem_ld_32x32(taddr + ch * kChunkCols + l * 32, *reinterpret_cast<uint32_t(*)[32]>(r + l * 32));
      tmem_ld_wait();
      if (ch == kChunks - 1) {                                  // last TMEM read of the tile: release the accumulator
        tc_fence_before();
        if (rank == 0) mbar_arrive(tmem_empty_bar);
        else mbar_arrive_cluster(tmem_empty_bar, 0);
      }
      if constexpr (kGather) {                                  // G_0 joins the accumulator registers, G_1 waits staged
        auto stage = [&]() {
#pragma unroll
          for (int t = 0; t < 8; ++t) sts_v4(((t & 1) ? coop_odd : coop_even) + (uint32_t)(t >> 1) * 1024u, gpre[t]);
          __syncwarp();
        };
        stage();
#pragma unroll
        for (int jp = 0; jp < 8; ++jp) {
          float a[kPer];
#pragma unroll
          for (int e = 0; e < kPer; ++e) a[e] = __uint_as_float(r[jp * kPer + e]);
          add_piece(a, lds_v4(my_row + (((uint32_t)jp ^ my_sw) << 4)));
#pragma unroll
          for (int e = 0; e < kPer; ++e) r[jp * kPer + e] = __float_as_uint(a[e]);
        }
        __syncwarp();
        if (p.n_gather > 1) { fetch_gather(1, ch); stage(); }
        if (ch + 1 < kChunks) fetch_gather(0, ch + 1);
      }
#pragma unroll
      for (int jp = 0; jp < 8; ++jp) {                          // 16-byte pieces of this thread's 128-byte row chunk
        const uint32_t addr = my_row + (((uint32_t)jp ^ my_sw) << 4);
        const int c0 = ch * kChunkCols + jp * kPer;
        float v[kPer];
        if constexpr (kGather) {                                // acc + G_0 + bias + G_1 before the activation
#pragma unroll
          for (int e = 0; e < kPer; ++e) v[e] = __uint_as_float(r[jp * kPer + e]) + p.bias[c0 + e];
          if (p.n_gather > 1) add_piece(v, lds_v4(addr));
#pragma unroll
          for (int e = 0; e < kPer; ++e) {
            v[e] = fmaf(v[e] * inv, p.scale[c0 + e], p.shift[c0 + e]);
            if (p.relu) v[e] = fmaxf(v[e], 0.f);
          }
        } else {
#pragma unroll
          for (int e = 0; e < kPer; ++e) {
            v[e] = fmaf((__uint_as_float(r[jp * kPer + e]) + p.bias[c0 + e]) * inv, p.scale[c0 + e], p.shift[c0 + e]);
            if (p.relu) v[e] = fmaxf(v[e], 0.f);
          }
        }
        if constexpr (kRes) {                                   // skip rows enter after the activation
          const uint4 ad = lds_v4(addr);
          const uint32_t au[4] = {ad.x, ad.y, ad.z, ad.w};
          if constexpr (kOut16) {
#pragma unroll
            for (int e = 0; e < 4; ++e) Pack16<TOut>::add2(v[2 * e], v[2 * e + 1], au[e]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) v[e] += __uint_as_float(au[e]);
          }
        }
        uint4 o;
        if constexpr (kOut16) {
          o.x = Pack16<TOut>::pack(v[0], v[1]); o.y = Pack16<TOut>::pack(v[2], v[3]);
          o.z = Pack16<TOut>::pack(v[4], v[5]); o.w = Pack16<TOut>::pack(v[6], v[7]);
        } else {
          o.x = __float_as_uint(v[0]); o.y = __float_as_uint(v[1]); o.z = __float_as_uint(v[2]); o.w = __float_as_uint(v[3]);
        }
        sts_v4(addr, o);
      }
      __syncwarp();
      // coalesced store: 4 rows x 128 B per instruction
      [[maybe_unused]] float cs[8];                             // kPool: this lane's 8 columns summed over its 8 rows
      if constexpr (kPool) {
#pragma unroll
        for (int e = 0; e < 8; ++e) cs[e] = 0.f;
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const uint4 o = lds_v4(((t & 1) ? coop_odd : coop_even) + (uint32_t)(t >> 1) * 1024u);
        if (t * 4 + r4 < rows_here) {
          if constexpr (kPool) {
            using P = Pack16<TOut>;
            cs[0] = P::add_lo(o.x, cs[0]); cs[1] = P::add_hi(o.x, cs[1]); cs[2] = P::add_lo(o.y, cs[2]); cs[3] = P::add_hi(o.y, cs[3]);
            cs[4] = P::add_lo(o.z, cs[4]); cs[5] = P::add_hi(o.z, cs[5]); cs[6] = P::add_lo(o.w, cs[6]); cs[7] = P::add_hi(o.w, cs[7]);
          }
          if (keep_rows) stg_v4(out_base + (size_t)t * 4 * out_row_bytes + ch * 128, o);
        }
      }
      if constexpr (kPool) {                                    // rows 4t + r4: add the four lane groups (butterfly)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], 8);
          cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], 16);
        }
        if (r4 < 2 && rows_here > 0) {                          // lane groups 0 and 1 write the two halves of 8 columns
          float4* dst = reinterpret_cast<float4*>(p.pool_sums + (size_t)(warp_row0 >> 5) * kW128 + ch * kChunkCols + piece * kPer);
          dst[r4] = r4 == 0 ? make_float4(cs[0], cs[1], cs[2], cs[3]) : make_float4(cs[4], cs[5], cs[6], cs[7]);
        }
      }
      __syncwarp();                                             // the staging tile is free for the next chunk
    }
  }
}

template <typename TOut, bool kRes, bool kPool, bool kMn = false, bool kGather = false>
__global__ void __launch_bounds__(kGemmThreads, 1)
k_gemm128(const __grid_constant__ Gemm128Params p) {
  static_assert(!kMn || (sizeof(TOut) == 4 && !kRes && !kPool && !kGather), "weight-gradient mode: fp32 partials, plain epilogue");
  constexpr int kStages = kG128Stages;
  extern __shared__ uint8_t gemm128_smem_raw[];
  const uint32_t smem_base = (smem_u32(gemm128_smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B wants 1024 B
  uint8_t* smem_gen = gemm128_smem_raw + (smem_base - smem_u32(gemm128_smem_raw));
  const uint32_t stages_u32 = smem_base;
  const uint32_t epi_u32 = stages_u32 + kStages * kG128StageBytes;
  constexpr int kEpiBytes = kEpiWarps * kEpiStageBytes;
  const uint32_t bars_u32 = epi_u32 + kEpiBytes;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + kStages * kG128StageBytes + kEpiBytes + kG128MiscBytes - 64);
  auto full_bar = [&](int s) { return bars_u32 + 8u * s; };
  auto empty_bar = [&](int s) { return bars_u32 + 8u * (kStages + s); };
  auto tmem_full_bar = [&](int b) { return bars_u32 + 8u * (2 * kStages + b); };       // b: accumulator 0 / 1
  auto tmem_empty_bar = [&](int b) { return bars_u32 + 8u * (2 * kStages + 2 + b); };

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const uint32_t rank = cluster_ctarank();
  const int tile0 = blockIdx.x >> 1;
  const int tile_stride = gridDim.x >> 1;

  // ---- one-time setup
  if (warp == 0 && elect_one()) {
    for (int s = 0; s < p.n_seg; ++s) { tma_prefetch_desc(&p.seg[s].a); tma_prefetch_desc(&p.seg[s].b); }
  }
  cluster_sync();                              // both CTAs resident before the paired TMEM alloc
  if (warp == 1) {
    if (elect_one()) {
      for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 2); mbar_init(empty_bar(s), 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(tmem_full_bar(b), 1); mbar_init(tmem_empty_bar(b), 2 * 4 * 32); }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<2>(smem_u32(tmem_slot), 2 * kW128);
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (warp == 0) {
    // ================================================================ TMA producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      for (int tile = tile0; tile < p.n_tiles; tile += tile_stride) {
        if constexpr (kMn) {                                    // node chunk `tile`: 128-byte column boxes x kblk nodes
          const int32_t cols_per_box = p.k_elems_per_block;     // 64 (16-bit) / 32 (tf32) values = 128 B
          const uint32_t box_bytes = (uint32_t)p.k_elems_per_block * 128u;
          const void* map_a = &p.seg[rank].a;                   // rank 0: agg, rank 1: x
          for (int kb = 0; kb < p.kblocks[0]; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, kTagEmpty);
            const uint32_t sa = stages_u32 + stage * kG128StageBytes;
            const int32_t node0 = (int32_t)((int64_t)tile * p.chunk_k + (int64_t)kb * p.k_elems_per_block);
            if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * kG128StageBytes);
            else mbar_arrive_cluster(full_bar(stage), 0);
            for (int j = 0; j < kW128 / cols_per_box; ++j)
              tma_load_2d_cg2(sa + j * box_bytes, map_a, full_bar(stage), j * cols_per_box, node0);
            for (int j = 0; j < kG128BRows / cols_per_box; ++j)
              tma_load_2d_cg2(sa + kATileBytes + j * box_bytes, &p.seg[0].b, full_bar(stage),
                              (int32_t)rank * kG128BRows + j * cols_per_box, node0);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
          continue;
        }
        const int32_t row0 = tile * (2 * kTileM) + (int32_t)rank * kTileM;
        for (int s = 0; s < p.n_seg; ++s) {
          for (int kb = 0; kb < p.kblocks[s]; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, kTagEmpty);
            const uint32_t sa = stages_u32 + stage * kG128StageBytes;
            const int32_t k0 = kb * p.k_elems_per_block;
            if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * kG128StageBytes);
            else mbar_arrive_cluster(full_bar(stage), 0);
            tma_load_2d_cg2(sa, &p.seg[s].a, full_bar(stage), k0, row0);
            tma_load_2d_cg2(sa + kATileBytes, &p.seg[s].b, full_bar(stage), k0, (int32_t)rank * kG128BRows);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1 && rank == 0) {
    // ================================================================ MMA issuer (leader CTA)
    const uint32_t idesc = umma_idesc(p.a_fmt, p.b_fmt, 2 * kTileM, kW128) | (kMn ? (3u << 15) : 0u);   // a/b MN-major
    const bool tf32 = p.a_fmt == 2;
    [[maybe_unused]] const uint32_t mn_lbo = (uint32_t)p.k_elems_per_block * 128u;  // bytes between 128-byte MN blocks
    [[maybe_unused]] const uint32_t mn_kstep = tf32 ? 1024u : 2048u;                // one UMMA K step: 8 / 16 nodes
    uint32_t stage = 0, phase = 0, it = 0;
    for (int tile = tile0; tile < p.n_tiles; tile += tile_stride, ++it) {
      const uint32_t b = it & 1u;
      mbar_wait(tmem_empty_bar(b), ((it >> 1) & 1u) ^ 1u, kTagTmemEmpty);   // warpgroup b drained this accumulator
      tc_fence_after();
      const uint32_t d = tmem_base + b * kW128;
      uint32_t first = 1;
      for (int s = 0; s < p.n_seg; ++s) {
        const int nkb = p.kblocks[s];
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full_bar(stage), phase, kTagFull);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t sa = stages_u32 + stage * kG128StageBytes;
            const uint32_t sb = sa + kATileBytes;
#pragma unroll
            for (int k = 0; k < kStageKBytes / 32; ++k) {
              const uint32_t acc = (first && k == 0) ? 0u : 1u;
              if constexpr (kMn) {
                const uint64_t da = umma_smem_desc_mn(sa + k * mn_kstep, mn_lbo, tf32);
                const uint64_t db = umma_smem_desc_mn(sb + k * mn_kstep, mn_lbo, tf32);
                if (tf32) umma<2, true>(d, da, db, idesc, acc);
                else umma<2, false>(d, da, db, idesc, acc);
              } else {
                if (tf32) umma<2, true>(d, umma_smem_desc(sa + k * 32), umma_smem_desc(sb + k * 32), idesc, acc);
                else umma<2, false>(d, umma_smem_desc(sa + k * 32), umma_smem_desc(sb + k * 32), idesc, acc);
              }
            }
            umma_commit<2>(empty_bar(stage));                   // smem slot reusable once these MMAs retire
            if (s == p.n_seg - 1 && kb == nkb - 1) umma_commit<2>(tmem_full_bar(b));
          }
          __syncwarp();
          first = 0;
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= kEpiFirstWarp && warp < kEpiFirstWarp + kEpiWarps) {
    // ================================================================ epilogue warps 4..11
    const int ew = warp - kEpiFirstWarp, g = ew >> 2;
    epilogue128_warp<TOut, kRes, kPool, kGather>(p, tmem_base, epi_u32 + (uint32_t)ew * kEpiStageBytes, tmem_full_bar(g),
                                        tmem_empty_bar(g), rank, tile0, tile_stride, g);
  }

  // ---- teardown
  tc_fence_before();
  cluster_sync();
  if (warp == 1) tmem_dealloc<2>(tmem_base, 2 * kW128);
}

// ------------------------------------------------------------------ host side
// [rows, k] row-major matrix, box = box_rows rows x 128 bytes of K, 128B swizzle, zero fill out of bounds
// (make_operand_map with a box height of choice: the weight tile of a CTA is 64 rows here)
static inline int make_operand_map_rows(CUtensorMap* map, const void* base, int64_t rows, int64_t k, int64_t ld,
                                        uint32_t fmt, uint32_t box_rows) {
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return BG_ERR_CUDA;
  const bool tf32 = fmt == 2;
  const int esz = tf32 ? 4 : 2;
  const CUtensorMapDataType dt = tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                      : (fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(kStageKBytes / esz), box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, (CUtensorMapL2promotion)BG_TMA_L2_PROMOTION, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? BG_OK : BG_ERR_CUDA;
}

template <typename TOut, bool kRes, bool kPool, bool kMn = false, bool kGather = false>
static int launch_gemm128(const Gemm128Params& p, cudaStream_t stream) {
  auto kern = k_gemm128<TOut, kRes, kPool, kMn, kGather>;
  static bool attr_set = false;
  if (!attr_set) {
    BG_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kG128SmemBytes));
    attr_set = true;
  }
  const int sms = gemm_sm_count();
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  cfg.gridDim = dim3((unsigned)(2 * min(p.n_tiles, sms / 2)));
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.numAttrs = 1;
  cfg.attrs = attr;
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = kG128SmemBytes;
  cfg.stream = stream;
  BG_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p));
  return BG_OK;
}

}  // namespace bg
