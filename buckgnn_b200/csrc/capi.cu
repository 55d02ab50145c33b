// C-ABI entry points of libbuckgnn_b200.so (declared in include/buckgnn_b200.h).
// Unity build: the kernels live in the .cuh files included here.
#include <cstdio>
#include <cstring>

#include "common.cuh"
#include "csr_build.cuh"
#include "aggregate.cuh"
#include "aggregate_window.cuh"
#include "encoder.cuh"
#include "gemm_tc.cuh"
#include "gemm128.cuh"
#include "pool_head.cuh"
#include "train.cuh"
#include "sag_pool.cuh"
#include "max_bwd.cuh"
#include "node_head.cuh"

namespace bg {

static thread_local char g_last_error[512] = "";

void set_last_cuda_error(cudaError_t e, const char* what, const char* file, int line) {
  snprintf(g_last_error, sizeof(g_last_error), "CUDA error %d (%s) at %s:%d: %s", (int)e,
           cudaGetErrorString(e), file, line, what);
}
static int fail(int code, const char* msg) {
  snprintf(g_last_error, sizeof(g_last_error), "%s", msg);
  return code;
}
// "<entry point>: <message>" for implementations shared by the 512- and 128-wide entry points
static int fail_in(int code, const char* fn, const char* msg) {
  snprintf(g_last_error, sizeof(g_last_error), "%s: %s", fn, msg);
  return code;
}

int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// SM partition for co-running kernels (bg_set_sm_partition): 0 = the whole device
static int g_gemm_sm_limit = 0, g_agg_sm_limit = 0;
int gemm_sm_count() { const int n = sm_count(); return (g_gemm_sm_limit > 0 && g_gemm_sm_limit < n) ? g_gemm_sm_limit : n; }
static int agg_sm_count() { const int n = sm_count(); return (g_agg_sm_limit > 0 && g_agg_sm_limit < n) ? g_agg_sm_limit : n; }

PFN_tensorMapEncodeTiled get_tensor_map_encoder() {
  static PFN_tensorMapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tensorMapEncodeTiled>(p);
  }
  return fn;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

template <typename T>
__global__ void k_cast_f32_16(const float* __restrict__ src, T* __restrict__ dst, int64_t n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = Pack16<T>::one(src[i]);
}
__global__ void k_split_tf32(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float v = src[i];
    const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    if (hi) hi[i] = h;
    lo[i] = v - h;
  }
}

// warp per row: the row's CSR slots get the row id; every slot also gets its own index; optionally
// nonempty[r, 0:64] = [1 if the row has entries else 0, 0, 0, ...]  (a K = 64 GEMM operand)
template <typename T>
__global__ void k_expand_rowptr(const int32_t* __restrict__ rowptr, int64_t n_rows, int32_t* __restrict__ row_of,
                                int32_t* __restrict__ iota, T* __restrict__ nonempty, int as_count) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); r < n_rows; r += n_warps) {
    const int32_t b = rowptr[r], e = rowptr[r + 1];
    if (row_of)
      for (int32_t i = b + lane; i < e; i += 32) { row_of[i] = (int32_t)r; iota[i] = i; }
    if (nonempty) {
      // as_count: the row's degree as three base-256 digits in columns 0..2 (weights 1, 256, 65536 on the host side):
      // every digit is exact in bf16 / fp16 / tf32 operands, a plain count above 256 / 2048 would be rounded
      const int32_t deg = e - b;
      float v0 = 0.f;
      if (as_count) { if (lane < 3) v0 = (float)((deg >> (8 * lane)) & (lane == 2 ? 0x7fff : 0xff)); }
      else if (lane == 0 && deg > 0) v0 = 1.f;
      if constexpr (sizeof(T) == 2) { nonempty[r * 64 + lane] = Pack16<T>::one(v0); nonempty[r * 64 + 32 + lane] = Pack16<T>::one(0.f); }
      else { nonempty[r * 64 + lane] = v0; nonempty[r * 64 + 32 + lane] = 0.f; }
    }
  }
}

template <typename T>
__global__ void k_add(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ c, T* __restrict__ out, int64_t n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = (float)a[i] + (float)b[i];
    if (c) v += (float)c[i];
    if constexpr (sizeof(T) == 2) out[i] = Pack16<T>::one(v); else out[i] = v;
  }
}

// device words -> pinned (UVA-mapped) host memory, written by the SMs: a result read-back that needs no copy
// engine (a cudaMemcpyAsync D2H can queue behind a large H2D transfer of the next batch)
__global__ void k_publish_words(const int32_t* __restrict__ src, volatile int32_t* __restrict__ dst_host, int n) {
  if ((int)threadIdx.x < n) dst_host[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}


// Compact wire format of an inference batch -> the PyG layout `BuckGNN.forward` takes (pipeline.py: WireBatch).
// One CTA per graph (grid-stride): its explicit edges int32 -> int64, then -- for graphs whose super node is implicit --
// the hub pairs (s, i), (i, s) for i = first node .. s-1 in order, exactly where `create_super_node`
// (reference Dataset_Preparation/VirtualEdgeCreate.py:106-111) appends them; and the `batch` id of its nodes.
__global__ void __launch_bounds__(256)
k_expand_wire(const int32_t* __restrict__ wire_edges, int64_t E_wire, const int64_t* __restrict__ node_ptr,
              const int64_t* __restrict__ wire_ptr, const int64_t* __restrict__ full_ptr, int64_t G, int64_t E_full,
              int64_t* __restrict__ edge_index, int64_t* __restrict__ batch) {
  for (int64_t g = blockIdx.x; g < G; g += gridDim.x) {
    const int64_t n0 = node_ptr[g], n1 = node_ptr[g + 1];
    const int64_t w0 = wire_ptr[g], w1 = wire_ptr[g + 1];
    const int64_t f0 = full_ptr[g], f1 = full_ptr[g + 1];
    for (int64_t i = threadIdx.x; i < w1 - w0; i += blockDim.x) {
      edge_index[f0 + i] = (int64_t)wire_edges[w0 + i];
      edge_index[E_full + f0 + i] = (int64_t)wire_edges[E_wire + w0 + i];
    }
    const int64_t hub_pairs = ((f1 - f0) - (w1 - w0)) / 2;          // 0, or n_g - 1: an implicit super node
    const int64_t s = n1 - 1, base = f0 + (w1 - w0);
    for (int64_t i = threadIdx.x; i < hub_pairs; i += blockDim.x) {
      edge_index[base + 2 * i] = s;              edge_index[E_full + base + 2 * i] = n0 + i;
      edge_index[base + 2 * i + 1] = n0 + i;     edge_index[E_full + base + 2 * i + 1] = s;
    }
    for (int64_t i = n0 + threadIdx.x; i < n1; i += blockDim.x) batch[i] = g;
  }
}

static inline int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }
static inline unsigned grid_for(int64_t n, int threads, int max_blocks) {
  int64_t b = ceil_div64(n > 0 ? n : 1, threads);
  return (unsigned)(b < max_blocks ? b : max_blocks);
}

struct HubRangeArgs { const int32_t* hub_lo; const int32_t* hub_of_row; int32_t max_degree; float* partial; };

template <typename T> static inline unsigned agg_grid(int64_t N) {
  return (unsigned)min64(ceil_div64(N, agg_row_threads<T>() / 32), (int64_t)agg_sm_count());
}
static inline int64_t hub_parts(int64_t band, int32_t max_degree) { return ceil_div64(max_degree > 0 ? max_degree : 1, band) + 1; }

template <typename T>
static int aggregate_dispatch(const T* x, T* out, int64_t N, const int32_t* rowptr, const int32_t* col,
                              const int32_t* big_rows, int32_t n_big, int aggr, float* partial, int32_t* ticket,
                              int width, const HubRangeArgs& hr, cudaStream_t stream) {
  if (width == 128) {
    const unsigned grid128 = (unsigned)min64(ceil_div64(N, 32), (int64_t)sm_count());
    const unsigned hub_grid128 = (unsigned)n_big * kHubSlices;
#define BG_AGG128_CASE(A)                                                                                        \
  case A:                                                                                                        \
    k_aggregate_rows128<T, A><<<grid128, 1024, 0, stream>>>(x, out, N, rowptr, col);                             \
    if (n_big > 0)                                                                                               \
      k_aggregate_hubs128<T, A><<<hub_grid128, kAggWarpsPerBlock * 32, 0, stream>>>(x, out, rowptr, col,         \
                                                                                    big_rows, n_big, partial, ticket); \
    break;
    switch (aggr) {
      BG_AGG128_CASE(BG_AGGR_MEAN)
      BG_AGG128_CASE(BG_AGGR_SUM)
      BG_AGG128_CASE(BG_AGGR_MAX)
      default: return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad aggr");
    }
#undef BG_AGG128_CASE
    BG_LAUNCH_OK();
    return BG_OK;
  }
  const unsigned grid = agg_grid<T>(N);
  const int64_t band = ceil_div64(N, grid);
  if constexpr (sizeof(T) == 2) {
    // 16-bit rows, opt-in (BG_AGG_WINDOW=1 in the environment): the band's rows staged once through a shared-memory ring
    // (aggregate_window.cuh).  Bit-identical results, but measured SLOWER than the L1/L2-gather kernels below (r02, cfg 2:
    // 0.59 vs 0.42 ms; stiffened degree-11 meshes 0.49 vs 0.41 ms per launch): the +-84-row window takes 21 of the ring's 27
    // slots, the 48 KB left in flight ahead of the gather front cannot cover HBM latency at 44 GB/s per SM.
    static const bool use_window = [] { const char* e = getenv("BG_AGG_WINDOW"); return e && e[0] == '1'; }();
    if (use_window) {
      const bool fold = hr.hub_lo && n_big > 0 && aggr != BG_AGGR_MAX;
      const HubFold hf = fold ? HubFold{hr.hub_of_row, hr.hub_lo, hr.partial, (int32_t)hub_parts(band, hr.max_degree)}
                              : HubFold{nullptr, nullptr, nullptr, 0};
#define BG_AGGW_LAUNCH(A, F)                                                                                          \
  {                                                                                                                   \
    static bool set = false;                                                                                          \
    if (!set) { BG_CUDA_OK(cudaFuncSetAttribute(k_aggregate_window<T, A, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWinSmemBytes)); set = true; } \
    k_aggregate_window<T, A, F><<<grid, kWinThreads, kWinSmemBytes, stream>>>(x, out, N, band, rowptr, col, hf);      \
  }
      if (fold) {
        if (aggr == BG_AGGR_MEAN) { BG_AGGW_LAUNCH(BG_AGGR_MEAN, true); k_hub_finalize<T, BG_AGGR_MEAN><<<(unsigned)n_big, 128, 0, stream>>>(out, N, band, rowptr, big_rows, hf); }
        else if (aggr == BG_AGGR_SUM) { BG_AGGW_LAUNCH(BG_AGGR_SUM, true); k_hub_finalize<T, BG_AGGR_SUM><<<(unsigned)n_big, 128, 0, stream>>>(out, N, band, rowptr, big_rows, hf); }
        else return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad aggr");
      } else {
        const unsigned hub_grid_w = (unsigned)n_big * kHubSlices;
        if (aggr == BG_AGGR_MEAN) { BG_AGGW_LAUNCH(BG_AGGR_MEAN, false); if (n_big > 0) k_aggregate_hubs<T, BG_AGGR_MEAN><<<hub_grid_w, kAggWarpsPerBlock * 32, 0, stream>>>(x, out, rowptr, col, big_rows, n_big, partial, ticket); }
        else if (aggr == BG_AGGR_SUM) { BG_AGGW_LAUNCH(BG_AGGR_SUM, false); if (n_big > 0) k_aggregate_hubs<T, BG_AGGR_SUM><<<hub_grid_w, kAggWarpsPerBlock * 32, 0, stream>>>(x, out, rowptr, col, big_rows, n_big, partial, ticket); }
        else if (aggr == BG_AGGR_MAX) { BG_AGGW_LAUNCH(BG_AGGR_MAX, false); if (n_big > 0) k_aggregate_hubs<T, BG_AGGR_MAX><<<hub_grid_w, kAggWarpsPerBlock * 32, 0, stream>>>(x, out, rowptr, col, big_rows, n_big, partial, ticket); }
        else return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad aggr");
      }
#undef BG_AGGW_LAUNCH
      BG_LAUNCH_OK();
      return BG_OK;
    }
  }
  if (hr.hub_lo && n_big > 0) {                    // range hubs folded into the row pass
    constexpr int kThreads = agg_fold_threads<T>();
    HubFold hf{hr.hub_of_row, hr.hub_lo, hr.partial, (int32_t)hub_parts(band, hr.max_degree)};
    constexpr int smem = agg_fold_smem<T>();
#define BG_AGGF_CASE(A)                                                                                              \
  case A: {                                                                                                          \
    static bool set = false;                                                                                         \
    if (!set) {                                                                                                      \
      BG_CUDA_OK(cudaFuncSetAttribute(k_aggregate_rows<T, A, true, kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
      /* the gathers live on the L1 window: ask for the smallest shared-memory carve-out that holds the stream ring */ \
      BG_CUDA_OK(cudaFuncSetAttribute(k_aggregate_rows<T, A, true, kThreads>, cudaFuncAttributePreferredSharedMemoryCarveout, \
                                      (smem + 1024) * 100 / (228 * 1024) + 1));                                      \
      set = true;                                                                                                    \
    }                                                                                                                \
    k_aggregate_rows<T, A, true, kThreads><<<grid, kThreads, smem, stream>>>(x, out, N, band, rowptr, col, hf);      \
    k_hub_finalize<T, A><<<(unsigned)n_big, 128, 0, stream>>>(out, N, band, rowptr, big_rows, hf);                   \
  } break;
    switch (aggr) {
      BG_AGGF_CASE(BG_AGGR_MEAN)
      BG_AGGF_CASE(BG_AGGR_SUM)
      default: return fail(BG_ERR_UNSUPPORTED, "bg_sage_aggregate: range hubs fold into mean / sum aggregation only");
    }
#undef BG_AGGF_CASE
    BG_LAUNCH_OK();
    return BG_OK;
  }
  const unsigned hub_grid = (unsigned)n_big * kHubSlices;
  const HubFold none{nullptr, nullptr, nullptr, 0};
#define BG_AGG_CASE(A)                                                                                       \
  case A:                                                                                                    \
    k_aggregate_rows<T, A, false, agg_row_threads<T>()><<<grid, agg_row_threads<T>(), 0, stream>>>(x, out, N, band, rowptr, col, none); \
    if (n_big > 0)                                                                                           \
      k_aggregate_hubs<T, A><<<hub_grid, kAggWarpsPerBlock * 32, 0, stream>>>(x, out, rowptr, col, big_rows, \
                                                                              n_big, partial, ticket);      \
    break;
  switch (aggr) {
    BG_AGG_CASE(BG_AGGR_MEAN)
    BG_AGG_CASE(BG_AGGR_SUM)
    BG_AGG_CASE(BG_AGGR_MAX)
    default: return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad aggr");
  }
#undef BG_AGG_CASE
  BG_LAUNCH_OK();
  return BG_OK;
}


template <typename T, int kW>
static void pool_launch(const T* x, const int32_t* graph_ptr, int64_t G, int mode, const float* pre_w, const float* pre_b,
                        const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                        const float* b3, int out_dim, float* pred, float* pooled_out, float* partial, const int32_t* nonfinite,
                        cudaStream_t stream) {
  if (mode != BG_POOL_SUPERNODE_ONLY) {
    dim3 grid((unsigned)G, kPoolSlices);
    const int exclude_last = (mode == BG_POOL_MEAN_NO_SUPER || mode == BG_POOL_SUPERNODE_WITH_POOLING) ? 1 : 0;
    k_pool_partial<T, kW><<<grid, kPoolWarps * 32, 0, stream>>>(x, graph_ptr, partial, exclude_last);
  }
  k_pool_head<T, kW><<<(unsigned)G, 128, 0, stream>>>(x, partial, graph_ptr, mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3,
                                                       out_dim, pred, pooled_out, nonfinite);
}

template <typename T, int kW>
static void pool_blocks_launch(const T* x, const int32_t* graph_ptr, int64_t G, int mode, const float* pre_w,
                               const float* pre_b, const float* w1, const float* b1, const float* w2, const float* b2,
                               const float* w3, const float* b3, int out_dim, float* pred, float* pooled_out,
                               const float* block_sums, const uint8_t* keep, float* partial, const int32_t* nonfinite,
                               cudaStream_t stream) {
  const int exclude_last = (mode == BG_POOL_MEAN_NO_SUPER || mode == BG_POOL_SUPERNODE_WITH_POOLING) ? 1 : 0;
  dim3 grid((unsigned)G, kPoolSlices);
  if (mode != BG_POOL_SUPERNODE_ONLY)
    k_pool_partial_blocks<T, kW><<<grid, kW / 2, 0, stream>>>(x, block_sums, keep, graph_ptr, partial, exclude_last);
  k_pool_head<T, kW><<<(unsigned)G, 128, 0, stream>>>(x, partial, graph_ptr, mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3,
                                                       out_dim, pred, pooled_out, nonfinite);
}

}  // namespace bg

using namespace bg;

template <typename T, int kW>
static void launch_max_bwd(const void* x, const void* agg, const void* dagg, int64_t N, const int32_t* rowptr_tgt,
                           const int32_t* col_tgt, const int32_t* big_tgt, int32_t n_big_tgt, const int32_t* rowptr_src,
                           const int32_t* col_src, const int32_t* big_src, int32_t n_big_src, void* w_scratch, void* dx,
                           float* partial, unsigned grid, cudaStream_t stream) {
  const T* xp = static_cast<const T*>(x); const T* ap = static_cast<const T*>(agg); const T* dp = static_cast<const T*>(dagg);
  T* wp = static_cast<T*>(w_scratch); T* op = static_cast<T*>(dx);
  // pass 1 (by target): w_i = dagg_i / n_i
  k_max_bwd_rows<T, 0, kW><<<grid, kMaxBwdWarps * 32, 0, stream>>>(ap, xp, nullptr, dp, rowptr_tgt, col_tgt, N, wp);
  if (n_big_tgt > 0) {
    k_max_bwd_big<T, 0, kW><<<dim3((unsigned)n_big_tgt, kMaxBwdSlices), kMaxBwdBigWarps * 32, 0, stream>>>(ap, xp, nullptr, rowptr_tgt, col_tgt, big_tgt, partial);
    k_max_bwd_big_finish<T, 0, kW><<<(unsigned)n_big_tgt, 32, 0, stream>>>(ap, dp, big_tgt, partial, wp);
  }
  // pass 2 (by source): dx_j = sum_i [agg_i == x_j] w_i
  k_max_bwd_rows<T, 1, kW><<<grid, kMaxBwdWarps * 32, 0, stream>>>(xp, ap, wp, nullptr, rowptr_src, col_src, N, op);
  if (n_big_src > 0) {
    k_max_bwd_big<T, 1, kW><<<dim3((unsigned)n_big_src, kMaxBwdSlices), kMaxBwdBigWarps * 32, 0, stream>>>(xp, ap, wp, rowptr_src, col_src, big_src, partial);
    k_max_bwd_big_finish<T, 1, kW><<<(unsigned)n_big_src, 32, 0, stream>>>(xp, nullptr, big_src, partial, op);
  }
}

extern "C" {

int bg_abi_version(void) { return BG_ABI_VERSION; }
const char* bg_last_error(void) { return g_last_error; }

int bg_device_check(void) {
  int dev = 0;
  BG_CUDA_OK(cudaGetDevice(&dev));
  int major = 0;
  BG_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return fail(BG_ERR_DEVICE, "buckgnn_b200 kernels are built for sm_100a only");
  return BG_OK;
}

#ifdef BG_PROFILE
// profiling build only: copy the per-CTA role cycle counters of the last bg_gemm512 to the host
int bg_gemm_prof_host(unsigned long long* out, int n) {
  BG_CUDA_OK(cudaMemcpyFromSymbol(out, g_gemm_prof, sizeof(unsigned long long) * (size_t)n));
  return BG_OK;
}
#endif

int bg_set_sm_partition(int gemm_sms, int agg_sms) {
  if (gemm_sms < 0 || agg_sms < 0 || gemm_sms == 1) return fail(BG_ERR_INVALID, "bg_set_sm_partition: bad SM count");
  g_gemm_sm_limit = gemm_sms;
  g_agg_sm_limit = agg_sms;
  return BG_OK;
}

int bg_watchdog_info_host(uint32_t* out4_host) {
  if (!out4_host) return fail(BG_ERR_INVALID, "null output");
  BG_CUDA_OK(cudaMemcpyFromSymbol(out4_host, g_watchdog_info, 16));
  return BG_OK;
}

// ------------------------------------------------------------------ K1
int64_t bg_csr_max_big_rows(int64_t n_edges) { return n_edges / (BG_BIG_ROW_THRESHOLD + 1) + 1; }

int bg_csr_workspace_bytes(int64_t n_nodes, int64_t n_edges, size_t* bytes_host) {
  if (!bytes_host || n_nodes < 0 || n_edges < 0) return fail(BG_ERR_INVALID, "bg_csr_workspace_bytes: bad argument");
  *bytes_host = csr_workspace_layout(nullptr, n_nodes).bytes;
  return BG_OK;
}

int bg_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int key_row,
                 int32_t* rowptr, int32_t* col, int32_t* perm, int32_t* big_rows, int32_t* info,
                 int32_t* hub_lo, int32_t* hub_of_row,
                 void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (E < 0 || N < 0 || E >= 0x7fffffffLL || N >= 0x7fffffffLL) return fail(BG_ERR_INVALID, "bg_csr_build: sizes out of range");
  if (key_row != 0 && key_row != 1) return fail(BG_ERR_INVALID, "bg_csr_build: key_row must be 0 or 1");
  if (!rowptr || !info || !workspace || (E > 0 && (!edge_index || !col || !perm || !big_rows)))
    return fail(BG_ERR_INVALID, "bg_csr_build: null pointer");
  CsrWorkspace w = csr_workspace_layout(workspace, N);
  if (workspace_bytes < w.bytes) return fail(BG_ERR_WORKSPACE, "bg_csr_build: workspace too small");
  const int64_t* key = edge_index + (size_t)key_row * E;
  const int64_t* other = edge_index + (size_t)(1 - key_row) * E;
  const int max_big = (int)bg_csr_max_big_rows(E);
  const int sms = sm_count();
  BG_CUDA_OK(cudaMemsetAsync(w.deg, 0, sizeof(int32_t) * (size_t)(N + 1), stream));
  if ((hub_lo != nullptr) != (hub_of_row != nullptr)) return fail(BG_ERR_INVALID, "bg_csr_build: hub_lo and hub_of_row go together");
  BG_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int32_t) * 2, stream));
  BG_CUDA_OK(cudaMemsetAsync(info + 4, 0, sizeof(int32_t) * 3, stream));
  BG_CUDA_OK(cudaMemsetAsync(rowptr, 0, sizeof(int32_t), stream));           // covers N == 0
  if (hub_of_row && N > 0) BG_CUDA_OK(cudaMemsetAsync(hub_of_row, 0xff, sizeof(int32_t) * (size_t)N, stream));
  if (N == 0) return BG_OK;
  if (E > 0) {
    k_csr_hist<<<grid_for(E, 256, sms * 16), 256, 0, stream>>>(key, E, N, w.deg, info);
    BG_LAUNCH_OK();
  }
  k_scan_block_sums<<<w.n_scan_blocks, 1024, 0, stream>>>(w.deg, N, w.block_sums);
  BG_LAUNCH_OK();
  k_scan_of_sums<<<1, 1024, 0, stream>>>(w.block_sums, w.n_scan_blocks);
  BG_LAUNCH_OK();
  k_scan_apply<<<w.n_scan_blocks, 1024, 0, stream>>>(w.deg, N, w.block_sums, rowptr, w.cursor, big_rows, info, max_big);
  BG_LAUNCH_OK();
  if (E > 0) {
    k_csr_fill<<<grid_for(E, 256, sms * 16), 256, 0, stream>>>(key, E, N, w.cursor, perm);
    BG_LAUNCH_OK();
    k_csr_sort_small<<<(unsigned)ceil_div64(N, 256), 256, 0, stream>>>(rowptr, N, other, perm, col, info);
    BG_LAUNCH_OK();
    static bool attr_set = false;
    const int sort_smem = kSortSmemElems * (int)sizeof(int32_t);
    if (!attr_set) {
      BG_CUDA_OK(cudaFuncSetAttribute(k_csr_sort_big, cudaFuncAttributeMaxDynamicSharedMemorySize, sort_smem));
      attr_set = true;
    }
    k_csr_sort_big<<<sms, 1024, sort_smem, stream>>>(rowptr, big_rows, info, max_big, other, N, perm, col, hub_lo, hub_of_row);
    BG_LAUNCH_OK();
  }
  return BG_OK;
}

int bg_batch_info(const int64_t* batch, int64_t N, int32_t* info, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!info || N < 0 || (N > 0 && !batch)) return fail(BG_ERR_INVALID, "bg_batch_info: bad argument");
  BG_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int32_t) * 2, stream));
  if (N == 0) return BG_OK;
  k_batch_info<<<grid_for(N, 256, sm_count() * 8), 256, 0, stream>>>(batch, N, info);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_graph_ptr_build(const int64_t* batch, int64_t N, int64_t G, int32_t* graph_ptr, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!graph_ptr || N < 0 || G < 0 || (N > 0 && !batch)) return fail(BG_ERR_INVALID, "bg_graph_ptr_build: bad argument");
  k_graph_ptr<<<grid_for(N + 1, 256, sm_count() * 8), 256, 0, stream>>>(batch, N, G, graph_ptr);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_publish_words(const int32_t* src, int32_t* dst_host_mapped, int32_t n, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!src || !dst_host_mapped || n <= 0 || n > 256) return fail(BG_ERR_INVALID, "bg_publish_words: bad argument");
  k_publish_words<<<1, 256, 0, stream>>>(src, dst_host_mapped, n);
  BG_LAUNCH_OK();
  return BG_OK;
}

// ------------------------------------------------------------------ K5 front
int bg_encoder_front(const float* x, int64_t N, int32_t F, const float* w1, const float* b1,
                     const float* w2, const float* b2, const int32_t* row_gather, void* out, int out_dtype,
                     int32_t* nonfinite_flag, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || F <= 0 || F > kEncMaxF) return fail(BG_ERR_UNSUPPORTED, "bg_encoder_front: need 0 < n_features <= 32");
  if (N == 0) return BG_OK;
  if (!x || !w1 || !b1 || !w2 || !b2 || !out || !aligned16(out)) return fail(BG_ERR_INVALID, "bg_encoder_front: bad pointer");
  const int smem = (int)sizeof(EncoderSmem);
  const unsigned grid = (unsigned)min64(ceil_div64(N, kEncRows), (int64_t)sm_count() * 3);
#define BG_ENC_CASE(T)                                                                                         \
  {                                                                                                            \
    static bool set = false;                                                                                   \
    if (!set) { BG_CUDA_OK(cudaFuncSetAttribute(k_encoder_front<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); set = true; } \
    k_encoder_front<T><<<grid, kEncThreads, smem, stream>>>(x, N, F, w1, b1, w2, b2, row_gather, static_cast<T*>(out)); \
  }
#define BG_ENC_MMA_CASE(T)                                                                                     \
  {                                                                                                            \
    const int msmem = (int)sizeof(EncoderMmaSmem);                                                             \
    static bool set = false;                                                                                   \
    if (!set) { BG_CUDA_OK(cudaFuncSetAttribute(k_encoder_front_mma<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, msmem)); set = true; } \
    const unsigned mgrid = (unsigned)min64(ceil_div64(N, 16 * kEncMmaWarps), (int64_t)sm_count() * 2);        \
    k_encoder_front_mma<T><<<mgrid, kEncMmaWarps * 32, msmem, stream>>>(x, N, F, w1, b1, w2, b2, row_gather, static_cast<T*>(out), nonfinite_flag); \
  }
  if (out_dtype == BG_BF16) BG_ENC_MMA_CASE(__nv_bfloat16)
  else if (out_dtype == BG_F16) BG_ENC_MMA_CASE(__half)
  else if (out_dtype == BG_F32) BG_ENC_CASE(float)
  else return fail(BG_ERR_INVALID, "bg_encoder_front: bad out_dtype");
#undef BG_ENC_MMA_CASE
#undef BG_ENC_CASE
  BG_LAUNCH_OK();
  return BG_OK;
}

// ------------------------------------------------------------------ K2
static size_t generic_hub_bytes(int32_t n_big) {
  return (size_t)n_big * kHubSlices * kHidden * sizeof(float) + (size_t)n_big * sizeof(int32_t) + 256;
}
int bg_aggregate_workspace_bytes(int32_t n_big, size_t* bytes_host) {
  if (!bytes_host || n_big < 0) return fail(BG_ERR_INVALID, "bg_aggregate_workspace_bytes: bad argument");
  *bytes_host = generic_hub_bytes(n_big);
  return BG_OK;
}

static size_t hubfold_bytes(int64_t N, int dtype, int32_t n_big, int32_t max_degree) {
  const unsigned grid = dtype == BG_F32 ? agg_grid<float>(N) : agg_grid<__half>(N);
  const int64_t band = ceil_div64(N > 0 ? N : 1, grid);
  return (size_t)n_big * (size_t)hub_parts(band, max_degree) * kMaxStreamWarps * kHidden * sizeof(float) + 256;
}
int bg_hubfold_workspace_bytes(int64_t N, int dtype, int32_t n_big, int32_t max_degree, size_t* bytes_host) {
  if (!bytes_host || n_big < 0 || N < 0 || max_degree < 0) return fail(BG_ERR_INVALID, "bg_hubfold_workspace_bytes: bad argument");
  const size_t a = generic_hub_bytes(n_big), b = hubfold_bytes(N, dtype, n_big, max_degree);
  *bytes_host = a > b ? a : b;
  return BG_OK;
}

int bg_sage_aggregate(const void* x, void* out, int dtype, int64_t N, int32_t width, const int32_t* rowptr,
                      const int32_t* col, const int32_t* big_rows, int32_t n_big, int aggr,
                      const int32_t* hub_lo, const int32_t* hub_of_row, int32_t hub_max_degree,
                      void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || n_big < 0) return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad size");
  if (width != 512 && width != 128) return fail(BG_ERR_UNSUPPORTED, "bg_sage_aggregate: width must be 512 or 128");
  if (N == 0) return BG_OK;
  if (!x || !out || !rowptr || !aligned16(x) || !aligned16(out)) return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad pointer");
  if ((hub_lo != nullptr) != (hub_of_row != nullptr)) return fail(BG_ERR_INVALID, "bg_sage_aggregate: hub_lo and hub_of_row go together");
  float* partial = nullptr;
  int32_t* ticket = nullptr;
  HubRangeArgs hr{nullptr, nullptr, 0, nullptr};
  if (n_big > 0) {
    const bool fold = hub_lo != nullptr && width == 512;
    size_t need = generic_hub_bytes(n_big);
    if (fold) { const size_t f = hubfold_bytes(N, dtype, n_big, hub_max_degree); if (f > need) need = f; }
    if (!workspace || workspace_bytes < need || !big_rows) return fail(BG_ERR_WORKSPACE, "bg_sage_aggregate: workspace too small");
    if (fold) {
      hr = HubRangeArgs{hub_lo, hub_of_row, hub_max_degree, static_cast<float*>(workspace)};
    } else {
      partial = static_cast<float*>(workspace);
      ticket = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + (size_t)n_big * kHubSlices * kHidden * sizeof(float));
      BG_CUDA_OK(cudaMemsetAsync(ticket, 0, sizeof(int32_t) * (size_t)n_big, stream));
    }
  }
  if (dtype == BG_BF16)
    return aggregate_dispatch(static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), N, rowptr, col,
                              big_rows, n_big, aggr, partial, ticket, width, hr, stream);
  if (dtype == BG_F16)
    return aggregate_dispatch(static_cast<const __half*>(x), static_cast<__half*>(out), N, rowptr, col,
                              big_rows, n_big, aggr, partial, ticket, width, hr, stream);
  if (dtype == BG_F32)
    return aggregate_dispatch(static_cast<const float*>(x), static_cast<float*>(out), N, rowptr, col, big_rows, n_big,
                              aggr, partial, ticket, width, hr, stream);
  return fail(BG_ERR_INVALID, "bg_sage_aggregate: bad dtype");
}

// ------------------------------------------------------------------ K3
static inline int umma_format_of(int dtype) { return dtype == BG_F16 ? 0 : (dtype == BG_BF16 ? 1 : (dtype == BG_F32 ? 2 : -1)); }

static int gemm512_impl(const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype, int b_dtype,
                        const bg_epilogue* epi, const bg_fused_aggregate* fuse, void* out, int out_dtype, int64_t ldo,
                        int cta_group, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!segs || n_seg < 1 || n_seg > BG_MAX_GEMM_SEGMENTS) return fail(BG_ERR_INVALID, "bg_gemm512: bad segment count");
  if (m < 0 || m >= 0x7fffffffLL) return fail(BG_ERR_INVALID, "bg_gemm512: bad m");
  if (m == 0) return BG_OK;
  const int a_fmt = umma_format_of(a_dtype), b_fmt = umma_format_of(b_dtype);
  if (a_fmt < 0 || b_fmt < 0 || a_fmt != b_fmt)
    return fail(BG_ERR_INVALID, "bg_gemm512: a_dtype and b_dtype must be the same (bf16, f16 or f32)");
  if (umma_format_of(out_dtype) < 0) return fail(BG_ERR_INVALID, "bg_gemm512: bad out_dtype");
  if (cta_group != 2) return fail(BG_ERR_UNSUPPORTED, "bg_gemm512: only cta_group = 2 is built");
  const bool tf32 = a_fmt == 2;
  const int esz = tf32 ? 4 : 2, osz = out_dtype == BG_F32 ? 4 : 2;
  const int kblk = kStageKBytes / esz;
  if (!out || !aligned16(out) || (ldo * osz) % 16 != 0 || ldo < kHidden) return fail(BG_ERR_INVALID, "bg_gemm512: bad out/ldo");
  GemmParams p;
  memset(&p, 0, sizeof(p));
  for (int s = 0; s < n_seg; ++s) {
    const bg_gemm_segment& g = segs[s];
    const bool gathered = fuse != nullptr && s == 0;      // the A operand of this segment is produced inside the kernel
    if ((!g.a && !gathered) || !g.b || g.k <= 0 || g.k % kblk != 0) return fail(BG_ERR_UNSUPPORTED, "bg_gemm512: k must be a positive multiple of 64 (16-bit) / 32 (tf32)");
    if ((!gathered && (!aligned16(g.a) || (g.lda * esz) % 16 != 0 || g.lda < g.k)) || !aligned16(g.b) || (g.ldb * esz) % 16 != 0 || g.ldb < g.k)
      return fail(BG_ERR_INVALID, "bg_gemm512: operand alignment / leading dimension");
    const int groups = g.b_groups > 1 ? g.b_groups : 1;
    if (groups != (segs[0].b_groups > 1 ? segs[0].b_groups : 1)) return fail(BG_ERR_INVALID, "bg_gemm512: segments disagree on b_groups");
    if (groups > 1 && m != (int64_t)groups * kHidden) return fail(BG_ERR_INVALID, "bg_gemm512: b_groups needs m == b_groups * 512");
    int rc = gathered ? BG_OK : make_operand_map(&p.seg[s].a, g.a, m, g.k, g.lda, (uint32_t)a_fmt);
    if (rc == BG_OK) rc = make_operand_map(&p.seg[s].b, g.b, (int64_t)groups * kHidden, g.k, g.ldb, (uint32_t)b_fmt);
    if (rc != BG_OK) return fail(rc, "bg_gemm512: cuTensorMapEncodeTiled failed");
    p.kblocks[s] = g.k / kblk;
  }
  p.n_seg = n_seg;
  p.b_group_tiles = segs[0].b_groups > 1 ? kHidden / (kTileM * cta_group) : 0;
  p.k_elems_per_block = kblk;
  p.a_fmt = (uint32_t)a_fmt; p.b_fmt = (uint32_t)b_fmt;
  p.n_tiles = (int32_t)ceil_div64(m, kTileM * cta_group);
  p.m = m;
  for (int i = 0; i < kHidden; ++i) { p.bias[i] = 0.f; p.scale[i] = 1.f; p.shift[i] = 0.f; }
  if (epi) {
    if (epi->residual && (!aligned16(epi->residual) || (epi->ldr * osz) % 16 != 0 || epi->ldr < kHidden))
      return fail(BG_ERR_INVALID, "bg_gemm512: bad residual/ldr");
    if (epi->bn_scale_host && !epi->bn_shift_host) return fail(BG_ERR_INVALID, "bg_gemm512: bn_scale without bn_shift");
    if (epi->bias_host) memcpy(p.bias, epi->bias_host, sizeof(float) * kHidden);
    if (epi->bn_scale_host) {
      memcpy(p.scale, epi->bn_scale_host, sizeof(float) * kHidden);
      memcpy(p.shift, epi->bn_shift_host, sizeof(float) * kHidden);
    }
    p.normalize = epi->normalize; p.relu = epi->relu;
    if (!epi->gather[0] && epi->gather[1]) return fail(BG_ERR_INVALID, "bg_gemm512: gather[1] without gather[0]");
    for (int k = 0; k < 2; ++k) {
      if (!epi->gather[k]) break;
      if (!epi->gather_idx[k] || !aligned16(epi->gather[k]) || (epi->gather_ld * osz) % 16 != 0 || epi->gather_ld < kHidden)
        return fail(BG_ERR_INVALID, "bg_gemm512: bad gather operand");
      p.gather[k] = epi->gather[k]; p.gidx[k] = epi->gather_idx[k];
      p.n_gather = k + 1;
    }
    p.gather_ld = epi->gather_ld;
    if (p.n_gather > 0 && (epi->normalize || epi->residual))
      return fail(BG_ERR_UNSUPPORTED, "bg_gemm512: gathered addends cannot be combined with normalize or residual");
    p.residual = epi->residual; p.ldr = epi->ldr;
    if (epi->inv_norm_out && !epi->normalize) return fail(BG_ERR_INVALID, "bg_gemm512: inv_norm_out needs normalize");
    p.inv_norm_out = epi->inv_norm_out;
    if ((epi->pool_block_sums != nullptr) != (epi->pool_block_keep != nullptr))
      return fail(BG_ERR_INVALID, "bg_gemm512: pool_block_sums and pool_block_keep go together");
    if (epi->pool_block_sums) {
      if (!epi->normalize || out_dtype == BG_F32 || epi->residual || p.n_gather > 0 || !aligned16(epi->pool_block_sums))
        return fail(BG_ERR_UNSUPPORTED, "bg_gemm512: the pool-fused epilogue needs normalize, a 16-bit output and no addends");
      p.pool_sums = epi->pool_block_sums; p.pool_keep = epi->pool_block_keep;
    }
  }
  for (int i = 0; i < kHidden / 2; ++i) {
    const __half2 sc = __floats2half2_rn(p.scale[2 * i], p.scale[2 * i + 1]);
    const __half2 sh = __floats2half2_rn(p.shift[2 * i], p.shift[2 * i + 1]);
    memcpy(&p.scale_h2[i], &sc, 4);
    memcpy(&p.shift_h2[i], &sh, 4);
  }
  p.out = out; p.ldo = ldo;
  if (fuse) {
    // fused SAGE layer: segment 0 = (aggregate of fuse->x, lin_l), K = 512, gathered in the kernel; 16-bit activations,
    // the normalize epilogue (with or without skip rows, or pool-fused)
    if (tf32 || out_dtype == BG_F32) return fail(BG_ERR_UNSUPPORTED, "bg_sage_fused512: 16-bit activations only");
    if (segs[0].k != kHidden || (segs[0].b_groups > 1)) return fail(BG_ERR_UNSUPPORTED, "bg_sage_fused512: segment 0 must be K = 512, one weight group");
    if (!fuse->x || !fuse->rowptr || (!fuse->col && m > 0) || !aligned16(fuse->x) || fuse->ldx != kHidden)
      return fail(BG_ERR_INVALID, "bg_sage_fused512: bad x / CSR (rows of x must be contiguous: ldx == 512)");
    if (fuse->aggr != BG_AGGR_MEAN && fuse->aggr != BG_AGGR_SUM) return fail(BG_ERR_UNSUPPORTED, "bg_sage_fused512: mean / sum aggregation only");
    if (fuse->n_big < 0 || (fuse->n_big > 0 && (!fuse->hub_agg || !fuse->big_rows || !aligned16(fuse->hub_agg))))
      return fail(BG_ERR_INVALID, "bg_sage_fused512: hub rows need hub_agg and big_rows");
    if (p.n_gather > 0 || !p.normalize) return fail(BG_ERR_UNSUPPORTED, "bg_sage_fused512: the SAGE update epilogue (normalize) only");
    p.fuse_x = fuse->x; p.fuse_ldx = fuse->ldx; p.fuse_rowptr = fuse->rowptr; p.fuse_col = fuse->col;
    p.fuse_hub_agg = fuse->hub_agg; p.fuse_big_rows = fuse->big_rows; p.fuse_n_big = fuse->n_big;
    p.fuse_mean = fuse->aggr == BG_AGGR_MEAN ? 1 : 0;
#define BG_FUSED_OUT(ADD, POOL)                                                                        \
  (out_dtype == BG_BF16 ? launch_gemm512<2, __nv_bfloat16, ADD, false, POOL, true>(p, stream)           \
                        : launch_gemm512<2, __half, ADD, false, POOL, true>(p, stream))
    if (p.pool_sums) return BG_FUSED_OUT(kAddNone, true);
    if (p.residual) return BG_FUSED_OUT(kAddResidual, false);
    return BG_FUSED_OUT(kAddNone, false);
#undef BG_FUSED_OUT
  }
  // "plain" epilogue: no normalize, no BatchNorm vectors -> the packed 16-bit pass 2 (exactly equivalent rounding)
  const bool plain = !p.normalize && !(epi && epi->bn_scale_host) && out_dtype != BG_F32;
#define BG_GEMM_OUT2(ADD, PLAIN)                                                               \
  (out_dtype == BG_BF16 ? launch_gemm512<2, __nv_bfloat16, ADD, PLAIN>(p, stream)              \
   : out_dtype == BG_F16 ? launch_gemm512<2, __half, ADD, PLAIN>(p, stream)                    \
                         : launch_gemm512<2, float, ADD, false>(p, stream))
#define BG_GEMM_OUT(ADD) (plain ? BG_GEMM_OUT2(ADD, true) : BG_GEMM_OUT2(ADD, false))
  if (p.pool_sums)
    return out_dtype == BG_BF16 ? launch_gemm512<2, __nv_bfloat16, kAddNone, false, true>(p, stream)
                                : launch_gemm512<2, __half, kAddNone, false, true>(p, stream);
  if (p.n_gather > 0) return BG_GEMM_OUT(kAddGather);
  if (p.residual) return BG_GEMM_OUT(kAddResidual);
  return BG_GEMM_OUT(kAddNone);
#undef BG_GEMM_OUT2
#undef BG_GEMM_OUT
}

int bg_gemm512(const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype, int b_dtype,
               const bg_epilogue* epi, void* out, int out_dtype, int64_t ldo, int cta_group, void* stream_) {
  return gemm512_impl(segs, n_seg, m, a_dtype, b_dtype, epi, nullptr, out, out_dtype, ldo, cta_group, stream_);
}

int bg_sage_fused512(const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype, int b_dtype,
                     const bg_epilogue* epi, const bg_fused_aggregate* fuse, void* out, int out_dtype, int64_t ldo,
                     void* stream_) {
  if (!fuse) return fail(BG_ERR_INVALID, "bg_sage_fused512: fused aggregate description missing");
  if (n_seg < 2) return fail(BG_ERR_INVALID, "bg_sage_fused512: needs the (aggregate, lin_l) and (x, lin_r) segments");
  return gemm512_impl(segs, n_seg, m, a_dtype, b_dtype, epi, fuse, out, out_dtype, ldo, 2, stream_);
}

// bg_gemm128 and bg_gemm128_gathered: the gathered addends are only accepted through the second entry point
static int gemm128_impl(const char* fn, bool gathered, const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype,
                        int b_dtype, const bg_epilogue* epi, void* out, int out_dtype, int64_t ldo, int cta_group,
                        void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  // every argument is checked before the first CUDA call
  if (!segs || n_seg < 1 || n_seg > BG_MAX_GEMM_SEGMENTS) return fail_in(BG_ERR_INVALID, fn, "bad segment count");
  if (m < 0 || m >= 0x7fffffffLL) return fail_in(BG_ERR_INVALID, fn, "bad m");
  const int a_fmt = umma_format_of(a_dtype), b_fmt = umma_format_of(b_dtype);
  if (a_fmt < 0 || b_fmt < 0 || a_fmt != b_fmt)
    return fail_in(BG_ERR_INVALID, fn, "a_dtype and b_dtype must be the same (bf16, f16 or f32)");
  if (umma_format_of(out_dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad out_dtype");
  if (cta_group != 2) return fail_in(BG_ERR_UNSUPPORTED, fn, "only cta_group = 2 is built");
  const bool tf32 = a_fmt == 2;
  const int esz = tf32 ? 4 : 2, osz = out_dtype == BG_F32 ? 4 : 2;
  const int kblk = kStageKBytes / esz;
  if (!out || !aligned16(out) || (ldo * osz) % 16 != 0 || ldo < kW128) return fail_in(BG_ERR_INVALID, fn, "bad out/ldo");
  for (int s = 0; s < n_seg; ++s) {
    const bg_gemm_segment& g = segs[s];
    if (!g.a || !g.b) return fail_in(BG_ERR_INVALID, fn, "null operand");
    if (g.k <= 0 || g.k % kblk != 0) return fail_in(BG_ERR_UNSUPPORTED, fn, "k must be a positive multiple of 64 (16-bit) / 32 (tf32)");
    if (g.b_groups > 1) return fail_in(BG_ERR_UNSUPPORTED, fn, "b_groups is not built at width 128");
    if (!aligned16(g.a) || (g.lda * esz) % 16 != 0 || g.lda < g.k || !aligned16(g.b) || (g.ldb * esz) % 16 != 0 || g.ldb < g.k)
      return fail_in(BG_ERR_INVALID, fn, "operand alignment / leading dimension");
  }
  int n_gather = 0;
  if (epi) {
    if (!gathered && (epi->gather[0] || epi->gather[1]))
      return fail_in(BG_ERR_UNSUPPORTED, fn, "gathered addends are not built here (use bg_gemm128_gathered)");
    if (gathered) {
      if (!epi->gather[0] && epi->gather[1]) return fail_in(BG_ERR_INVALID, fn, "gather[1] without gather[0]");
      for (int k = 0; k < 2 && epi->gather[k]; ++k) {
        if (!epi->gather_idx[k] || !aligned16(epi->gather[k]) || epi->gather_ld < kW128 || (epi->gather_ld * osz) % 16 != 0)
          return fail_in(BG_ERR_INVALID, fn, "bad gather operand (null index, misaligned, or gather_ld < 128 / rows not 16-byte aligned)");
        n_gather = k + 1;
      }
      if (n_gather > 0 && (epi->normalize || epi->residual || epi->pool_block_sums || epi->pool_block_keep))
        return fail_in(BG_ERR_UNSUPPORTED, fn, "gathered addends cannot be combined with normalize, residual or pool fusion");
    }
    if (epi->residual && (!aligned16(epi->residual) || (epi->ldr * osz) % 16 != 0 || epi->ldr < kW128))
      return fail_in(BG_ERR_INVALID, fn, "bad residual/ldr");
    if (epi->bn_scale_host && !epi->bn_shift_host) return fail_in(BG_ERR_INVALID, fn, "bn_scale without bn_shift");
    if (epi->inv_norm_out && !epi->normalize) return fail_in(BG_ERR_INVALID, fn, "inv_norm_out needs normalize");
    if ((epi->pool_block_sums != nullptr) != (epi->pool_block_keep != nullptr))
      return fail_in(BG_ERR_INVALID, fn, "pool_block_sums and pool_block_keep go together");
    if (epi->pool_block_sums && (!epi->normalize || out_dtype == BG_F32 || epi->residual || !aligned16(epi->pool_block_sums)))
      return fail_in(BG_ERR_UNSUPPORTED, fn, "the pool-fused epilogue needs normalize, a 16-bit output and no residual");
  }
  if (m == 0) return BG_OK;
  Gemm128Params p;
  memset(&p, 0, sizeof(p));
  for (int s = 0; s < n_seg; ++s) {
    const bg_gemm_segment& g = segs[s];
    int rc = make_operand_map(&p.seg[s].a, g.a, m, g.k, g.lda, (uint32_t)a_fmt);
    if (rc == BG_OK) rc = make_operand_map_rows(&p.seg[s].b, g.b, kW128, g.k, g.ldb, (uint32_t)b_fmt, kG128BRows);
    if (rc != BG_OK) return fail_in(rc, fn, "cuTensorMapEncodeTiled failed");
    p.kblocks[s] = g.k / kblk;
  }
  p.n_seg = n_seg;
  p.k_elems_per_block = kblk;
  p.a_fmt = (uint32_t)a_fmt; p.b_fmt = (uint32_t)b_fmt;
  p.n_tiles = (int32_t)ceil_div64(m, 2 * kTileM);
  p.m = m;
  for (int i = 0; i < kW128; ++i) { p.bias[i] = 0.f; p.scale[i] = 1.f; p.shift[i] = 0.f; }
  if (epi) {
    if (epi->bias_host) memcpy(p.bias, epi->bias_host, sizeof(float) * kW128);
    if (epi->bn_scale_host) {
      memcpy(p.scale, epi->bn_scale_host, sizeof(float) * kW128);
      memcpy(p.shift, epi->bn_shift_host, sizeof(float) * kW128);
    }
    p.normalize = epi->normalize; p.relu = epi->relu;
    p.residual = epi->residual; p.ldr = epi->ldr;
    p.inv_norm_out = epi->inv_norm_out;
    p.pool_sums = epi->pool_block_sums; p.pool_keep = epi->pool_block_keep;
    for (int k = 0; k < n_gather; ++k) { p.gather[k] = epi->gather[k]; p.gidx[k] = epi->gather_idx[k]; }
    p.n_gather = n_gather;
    p.gather_ld = epi->gather_ld;
  }
  p.out = out; p.ldo = ldo;
  if (p.pool_sums)
    return out_dtype == BG_BF16 ? launch_gemm128<__nv_bfloat16, false, true>(p, stream)
                                : launch_gemm128<__half, false, true>(p, stream);
  if (n_gather > 0)
    return out_dtype == BG_BF16 ? launch_gemm128<__nv_bfloat16, false, false, false, true>(p, stream)
         : out_dtype == BG_F16  ? launch_gemm128<__half, false, false, false, true>(p, stream)
                                : launch_gemm128<float, false, false, false, true>(p, stream);
#define BG_GEMM128_OUT(RES)                                                              \
  (out_dtype == BG_BF16 ? launch_gemm128<__nv_bfloat16, RES, false>(p, stream)           \
   : out_dtype == BG_F16 ? launch_gemm128<__half, RES, false>(p, stream)                 \
                         : launch_gemm128<float, RES, false>(p, stream))
  return p.residual ? BG_GEMM128_OUT(true) : BG_GEMM128_OUT(false);
#undef BG_GEMM128_OUT
}

int bg_gemm128(const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype, int b_dtype,
               const bg_epilogue* epi, void* out, int out_dtype, int64_t ldo, int cta_group, void* stream_) {
  return gemm128_impl("bg_gemm128", false, segs, n_seg, m, a_dtype, b_dtype, epi, out, out_dtype, ldo, cta_group, stream_);
}

int bg_gemm128_gathered(const bg_gemm_segment* segs, int32_t n_seg, int64_t m, int a_dtype, int b_dtype,
                        const bg_epilogue* epi, void* out, int out_dtype, int64_t ldo, int cta_group, void* stream_) {
  return gemm128_impl("bg_gemm128_gathered", true, segs, n_seg, m, a_dtype, b_dtype, epi, out, out_dtype, ldo, cta_group,
                      stream_);
}

int bg_sage_aggregate_hubs(const void* x, int dtype, const int32_t* rowptr, const int32_t* col, const int32_t* big_rows,
                           int32_t n_big, int aggr, void* hub_out, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n_big < 0) return fail(BG_ERR_INVALID, "bg_sage_aggregate_hubs: bad n_big");
  if (n_big == 0) return BG_OK;
  if (!x || !rowptr || !col || !big_rows || !hub_out || !aligned16(x) || !aligned16(hub_out))
    return fail(BG_ERR_INVALID, "bg_sage_aggregate_hubs: bad pointer");
  if (!workspace || workspace_bytes < generic_hub_bytes(n_big)) return fail(BG_ERR_WORKSPACE, "bg_sage_aggregate_hubs: workspace too small");
  float* partial = static_cast<float*>(workspace);
  int32_t* ticket = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + (size_t)n_big * kHubSlices * kHidden * sizeof(float));
  BG_CUDA_OK(cudaMemsetAsync(ticket, 0, sizeof(int32_t) * (size_t)n_big, stream));
  const unsigned grid = (unsigned)n_big * kHubSlices;
#define BG_HUBS_CASE(T, A) k_aggregate_hubs<T, A, true><<<grid, kAggWarpsPerBlock * 32, 0, stream>>>(                 \
      static_cast<const T*>(x), static_cast<T*>(hub_out), rowptr, col, big_rows, n_big, partial, ticket)
  if (aggr != BG_AGGR_MEAN && aggr != BG_AGGR_SUM) return fail(BG_ERR_UNSUPPORTED, "bg_sage_aggregate_hubs: mean / sum only");
  if (dtype == BG_F16) { if (aggr == BG_AGGR_MEAN) BG_HUBS_CASE(__half, BG_AGGR_MEAN); else BG_HUBS_CASE(__half, BG_AGGR_SUM); }
  else if (dtype == BG_BF16) { if (aggr == BG_AGGR_MEAN) BG_HUBS_CASE(__nv_bfloat16, BG_AGGR_MEAN); else BG_HUBS_CASE(__nv_bfloat16, BG_AGGR_SUM); }
  else return fail(BG_ERR_UNSUPPORTED, "bg_sage_aggregate_hubs: 16-bit rows only");
#undef BG_HUBS_CASE
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_wgrad512(const void* dz, int64_t ld_dz, const void* act, int32_t act_cols, int64_t ld_act, int dtype, int64_t n_rows,
                int32_t n_chunks, int64_t chunk_k, float* partial, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int fmt = umma_format_of(dtype);
  if (fmt < 0) return fail(BG_ERR_INVALID, "bg_wgrad512: bad dtype");
  if (act_cols <= 0 || act_cols > kHidden || act_cols % 8 != 0) return fail(BG_ERR_INVALID, "bg_wgrad512: act_cols must be a multiple of 8 in (0, 512]");
  const int esz = fmt == 2 ? 4 : 2;
  const int kblk = kStageKBytes / esz;                     // nodes per pipeline stage: 64 (16-bit) / 32 (tf32)
  if (n_rows <= 0 || n_chunks <= 0 || chunk_k <= 0 || chunk_k % kblk != 0 || (int64_t)n_chunks * chunk_k < n_rows ||
      (int64_t)n_chunks * chunk_k >= 0x7fffffffLL)
    return fail(BG_ERR_INVALID, "bg_wgrad512: chunk_k must be a multiple of 64 (16-bit) / 32 (tf32) and n_chunks*chunk_k >= n_rows");
  if (!dz || !act || !partial || !aligned16(dz) || !aligned16(act) || !aligned16(partial) || ld_dz < kHidden ||
      ld_act < act_cols || (ld_dz * esz) % 16 != 0 || (ld_act * esz) % 16 != 0)
    return fail(BG_ERR_INVALID, "bg_wgrad512: bad pointer / leading dimension");
  GemmParams p;
  memset(&p, 0, sizeof(p));
  int rc = make_mn_operand_map(&p.seg[0].a, dz, n_rows, kHidden, ld_dz, (uint32_t)fmt, kblk);
  if (rc == BG_OK) rc = make_mn_operand_map(&p.seg[0].b, act, n_rows, act_cols, ld_act, (uint32_t)fmt, kblk);
  if (rc != BG_OK) return fail(rc, "bg_wgrad512: cuTensorMapEncodeTiled failed");
  p.n_seg = 1;
  p.kblocks[0] = (int32_t)(chunk_k / kblk);
  p.k_elems_per_block = kblk;
  p.a_fmt = p.b_fmt = (uint32_t)fmt;
  p.mn_major = 1;
  p.chunk_k = chunk_k;
  p.n_tiles = 2 * n_chunks;
  p.m = (int64_t)n_chunks * kHidden;
  for (int i = 0; i < kHidden; ++i) { p.bias[i] = 0.f; p.scale[i] = 1.f; p.shift[i] = 0.f; }
  p.out = partial; p.ldo = kHidden;
  return launch_gemm512<2, float, kAddNone, false>(p, stream);
}

// The weight-gradient GEMM of both 128-wide entry points: per node chunk one M = 256 pair tile [a0^T ; a1^T]·dz into
// partial.  `a1` null (a single product): the rank-1 CTA re-reads a0 (its rows arrive from L2 with rank 0's) and that
// half of the tile is discarded by the reduction.  Checks every argument it takes before any CUDA call; the callers
// check theirs before calling it.
static int wgrad128_gemm(const char* fn, const void* dz, const void* a0, const void* a1, int dtype, int64_t n_rows,
                         int32_t n_chunks, int64_t chunk_k, float* partial, cudaStream_t stream) {
  const int fmt = umma_format_of(dtype);
  if (fmt < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");
  const int esz = fmt == 2 ? 4 : 2;
  const int kblk = kStageKBytes / esz;                     // nodes per pipeline stage: 64 (16-bit) / 32 (tf32)
  if (n_rows <= 0 || n_chunks <= 0 || chunk_k <= 0 || chunk_k % kblk != 0 || (int64_t)n_chunks * chunk_k < n_rows ||
      (int64_t)n_chunks * chunk_k >= 0x7fffffffLL)
    return fail_in(BG_ERR_INVALID, fn, "chunk_k must be a multiple of 64 (16-bit) / 32 (tf32) and n_chunks*chunk_k >= n_rows");
  if (!dz || !a0 || !partial || !aligned16(dz) || !aligned16(a0) || (a1 && !aligned16(a1)) || !aligned16(partial))
    return fail_in(BG_ERR_INVALID, fn, "null or misaligned pointer");
  Gemm128Params p;
  memset(&p, 0, sizeof(p));
  int rc = make_mn_operand_map(&p.seg[0].a, a0, n_rows, kW128, kW128, (uint32_t)fmt, kblk);
  if (rc == BG_OK) rc = make_mn_operand_map(&p.seg[1].a, a1 ? a1 : a0, n_rows, kW128, kW128, (uint32_t)fmt, kblk);
  if (rc == BG_OK) rc = make_mn_operand_map(&p.seg[0].b, dz, n_rows, kW128, kW128, (uint32_t)fmt, kblk);
  if (rc != BG_OK) return fail_in(rc, fn, "cuTensorMapEncodeTiled failed");
  p.n_seg = 1;                                             // the MMA warp walks segment 0's K blocks; rank 1 reads seg[1].a
  p.kblocks[0] = (int32_t)(chunk_k / kblk);
  p.k_elems_per_block = kblk;
  p.a_fmt = p.b_fmt = (uint32_t)fmt;
  p.chunk_k = chunk_k;
  p.n_tiles = n_chunks;
  p.m = (int64_t)n_chunks * 2 * kW128;
  for (int i = 0; i < kW128; ++i) { p.bias[i] = 0.f; p.scale[i] = 1.f; p.shift[i] = 0.f; }
  p.out = partial; p.ldo = kW128;
  return launch_gemm128<float, false, false, true>(p, stream);
}

int bg_wgrad128(const void* dz, const void* agg, const void* x, int dtype, int64_t n_rows, int32_t n_chunks, int64_t chunk_k,
                float* partial, float* dwl, float* dwr, int accumulate, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!agg || !x || !dwl || !dwr) return fail(BG_ERR_INVALID, "bg_wgrad128: null or misaligned pointer");
  const int rc = wgrad128_gemm("bg_wgrad128", dz, agg, x, dtype, n_rows, n_chunks, chunk_k, partial, stream);
  if (rc != BG_OK) return rc;
  k_reduce_wgrad128<<<grid_for(2 * kW128 * kW128, 256, sm_count() * 4), 256, 0, stream>>>(partial, n_chunks, dwl, dwr, accumulate);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_wgrad128_ld(const void* dz, const void* a0, const void* a1, int dtype, int64_t n_rows, int32_t n_chunks, int64_t chunk_k,
                   float* partial, float* dw0, int64_t ld0, float* dw1, int64_t ld1, int accumulate, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!dw0 || ld0 < kW128 || (a1 && (!dw1 || ld1 < kW128)) || (!a1 && dw1))
    return fail(BG_ERR_INVALID, "bg_wgrad128_ld: dw0 (and dw1 exactly when a1 is given) non-null with ld >= 128");
  const int rc = wgrad128_gemm("bg_wgrad128_ld", dz, a0, a1, dtype, n_rows, n_chunks, chunk_k, partial, stream);
  if (rc != BG_OK) return rc;
  k_reduce_wgrad128_ld<<<grid_for((a1 ? 2 : 1) * kW128 * kW128, 256, sm_count() * 4), 256, 0, stream>>>(
      partial, n_chunks, dw0, ld0, a1 ? dw1 : nullptr, ld1, accumulate);
  BG_LAUNCH_OK();
  return BG_OK;
}

// ------------------------------------------------------------------ K4
int bg_pool_workspace_bytes(int64_t G, size_t* bytes_host) {
  if (!bytes_host || G < 0) return fail(BG_ERR_INVALID, "bg_pool_workspace_bytes: bad argument");
  *bytes_host = (size_t)G * kPoolSlices * kHidden * sizeof(float) + 256;
  return BG_OK;
}

static int pool_head_impl(const char* fn, int width, const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                 const float* pre_w, const float* pre_b,
                 const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                 int32_t out_dim, float* pred, float* pooled_out, void* workspace, size_t workspace_bytes,
                 const int32_t* nonfinite_flag, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G < 0 || N < 0 || G > 65535LL * 1024) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (G == 0) return BG_OK;
  if (out_dim < 1 || out_dim > 64) return fail_in(BG_ERR_UNSUPPORTED, fn, "out_dim must be in [1,64]");
  if (pool_mode < BG_POOL_MEAN || pool_mode > BG_POOL_SUPERNODE_WITH_POOLING) return fail_in(BG_ERR_INVALID, fn, "bad pool_mode");
  if ((pre_w != nullptr) != (pre_b != nullptr) || (pre_w && pool_mode > BG_POOL_MEAN_NO_SUPER) || (pre_w && !aligned16(pre_w)))
    return fail_in(BG_ERR_INVALID, fn, "pooling MLP needs both pre_w and pre_b and a mean pooling mode");
  if (!graph_ptr || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !pred || (N > 0 && (!x || !aligned16(x))) || !aligned16(w1))
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  size_t need = 0;
  bg_pool_workspace_bytes(G, &need);
  if (!workspace || workspace_bytes < need) return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  float* partial = static_cast<float*>(workspace);
  if (dtype == BG_BF16)
    (width == kHidden ? pool_launch<__nv_bfloat16, kHidden> : pool_launch<__nv_bfloat16, kW128>)(
        static_cast<const __nv_bfloat16*>(x), graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim, pred, pooled_out, partial, nonfinite_flag, stream);
  else if (dtype == BG_F16)
    (width == kHidden ? pool_launch<__half, kHidden> : pool_launch<__half, kW128>)(
        static_cast<const __half*>(x), graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim, pred, pooled_out, partial, nonfinite_flag, stream);
  else if (dtype == BG_F32)
    (width == kHidden ? pool_launch<float, kHidden> : pool_launch<float, kW128>)(
        static_cast<const float*>(x), graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim, pred, pooled_out, partial, nonfinite_flag, stream);
  else
    return fail_in(BG_ERR_INVALID, fn, "bad dtype");
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_pool_head(const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                 const float* pre_w, const float* pre_b,
                 const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                 int32_t out_dim, float* pred, float* pooled_out, void* workspace, size_t workspace_bytes,
                 const int32_t* nonfinite_flag, void* stream_) {
  return pool_head_impl("bg_pool_head", kHidden, x, dtype, N, graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3,
                        out_dim, pred, pooled_out, workspace, workspace_bytes, nonfinite_flag, stream_);
}

int bg_pool_head128(const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                    const float* pre_w, const float* pre_b,
                    const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                    int32_t out_dim, float* pred, float* pooled_out, void* workspace, size_t workspace_bytes,
                    const int32_t* nonfinite_flag, void* stream_) {
  return pool_head_impl("bg_pool_head128", kW128, x, dtype, N, graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3,
                        b3, out_dim, pred, pooled_out, workspace, workspace_bytes, nonfinite_flag, stream_);
}

int bg_pool_block_flags(const int32_t* graph_ptr, int64_t G, int64_t N, uint8_t* keep, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G < 0 || N < 0 || !graph_ptr || (N > 0 && !keep)) return fail(BG_ERR_INVALID, "bg_pool_block_flags: bad argument");
  if (N == 0) return BG_OK;
  BG_CUDA_OK(cudaMemsetAsync(keep, 0, (size_t)ceil_div64(N, 32), stream));
  k_pool_block_flags<<<(unsigned)ceil_div64(G + 1, 256), 256, 0, stream>>>(graph_ptr, G, N, keep);
  BG_LAUNCH_OK();
  return BG_OK;
}

static int pool_head_blocks_impl(const char* fn, int width, const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                        const float* pre_w, const float* pre_b,
                        const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                        int32_t out_dim, float* pred, float* pooled_out, const float* block_sums, const uint8_t* keep,
                        void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G < 0 || N < 0 || G > 65535LL * 1024) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (G == 0) return BG_OK;
  if (out_dim < 1 || out_dim > 64) return fail_in(BG_ERR_UNSUPPORTED, fn, "out_dim must be in [1,64]");
  if (pool_mode < BG_POOL_MEAN || pool_mode > BG_POOL_SUPERNODE_WITH_POOLING) return fail_in(BG_ERR_INVALID, fn, "bad pool_mode");
  if ((pre_w != nullptr) != (pre_b != nullptr) || (pre_w && pool_mode > BG_POOL_MEAN_NO_SUPER) || (pre_w && !aligned16(pre_w)))
    return fail_in(BG_ERR_INVALID, fn, "pooling MLP needs both pre_w and pre_b and a mean pooling mode");
  if (!graph_ptr || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !pred || !aligned16(w1) ||
      (N > 0 && (!x || !aligned16(x) || !block_sums || !aligned16(block_sums) || !keep)))
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  if (dtype != BG_BF16 && dtype != BG_F16) return fail_in(BG_ERR_UNSUPPORTED, fn, "16-bit rows only");
  size_t need = 0;
  bg_pool_workspace_bytes(G, &need);
  if (!workspace || workspace_bytes < need) return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  float* partial = static_cast<float*>(workspace);
  if (dtype == BG_BF16)
    (width == kHidden ? pool_blocks_launch<__nv_bfloat16, kHidden> : pool_blocks_launch<__nv_bfloat16, kW128>)(
        static_cast<const __nv_bfloat16*>(x), graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim, pred, pooled_out, block_sums, keep, partial, nonfinite_flag, stream);
  else
    (width == kHidden ? pool_blocks_launch<__half, kHidden> : pool_blocks_launch<__half, kW128>)(
        static_cast<const __half*>(x), graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim, pred, pooled_out, block_sums, keep, partial, nonfinite_flag, stream);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_pool_head_blocks(const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                        const float* pre_w, const float* pre_b,
                        const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                        int32_t out_dim, float* pred, float* pooled_out, const float* block_sums, const uint8_t* keep,
                        void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream_) {
  return pool_head_blocks_impl("bg_pool_head_blocks", kHidden, x, dtype, N, graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1,
                               w2, b2, w3, b3, out_dim, pred, pooled_out, block_sums, keep, workspace, workspace_bytes,
                               nonfinite_flag, stream_);
}

int bg_pool_head_blocks128(const void* x, int dtype, int64_t N, const int32_t* graph_ptr, int64_t G, int pool_mode,
                           const float* pre_w, const float* pre_b,
                           const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                           int32_t out_dim, float* pred, float* pooled_out, const float* block_sums, const uint8_t* keep,
                           void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream_) {
  return pool_head_blocks_impl("bg_pool_head_blocks128", kW128, x, dtype, N, graph_ptr, G, pool_mode, pre_w, pre_b, w1, b1,
                               w2, b2, w3, b3, out_dim, pred, pooled_out, block_sums, keep, workspace, workspace_bytes,
                               nonfinite_flag, stream_);
}

// ------------------------------------------------------------------ node-level head, hidden_channels = 128
int bg_node_head128(const void* x, int dtype, int64_t n_rows, const void* w1, const float* b1, const float* w2,
                    const float* b2, int32_t out_dim, float* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dtype != BG_BF16 && dtype != BG_F16 && dtype != BG_F32) return fail(BG_ERR_INVALID, "bg_node_head128: bad dtype");
  if (n_rows < 0) return fail(BG_ERR_INVALID, "bg_node_head128: n_rows < 0");
  if (out_dim < 1 || out_dim > kNhMaxOut) return fail(BG_ERR_INVALID, "bg_node_head128: out_dim must be in 1..8");
  if (!w1 || !b1 || !w2 || !b2 || !aligned16(w1) || !aligned4(b1) || !aligned4(w2) || !aligned4(b2))
    return fail(BG_ERR_INVALID, "bg_node_head128: bad weight pointer (null, or w1 not 16-byte / b1, w2, b2 not 4-byte aligned)");
  // x and out may be null only when there are no rows (an empty tensor has no storage)
  if ((n_rows > 0 && (!x || !out)) || !aligned16(x) || !aligned4(out))
    return fail(BG_ERR_INVALID, "bg_node_head128: bad x / out pointer (null, or x not 16-byte / out not 4-byte aligned)");
  if (n_rows == 0) return BG_OK;
  if (dtype == BG_F32) {
    const int smem = (int)sizeof(NodeHeadSmem32);
    static bool set = false;
    if (!set) { BG_CUDA_OK(cudaFuncSetAttribute(k_node_head128_f32, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); set = true; }
    const unsigned grid = (unsigned)min64(ceil_div64(n_rows, kNhRows32), (int64_t)sm_count() * 2);
    k_node_head128_f32<<<grid, 256, smem, stream>>>(static_cast<const float*>(x), n_rows, static_cast<const float*>(w1),
                                                    b1, w2, b2, out_dim, out);
  } else {
    const unsigned grid = (unsigned)min64(ceil_div64(n_rows, 16 * kNhWarps), (int64_t)sm_count() * 2);
    if (dtype == BG_BF16)
      k_node_head128_mma<__nv_bfloat16><<<grid, kNhWarps * 32, 0, stream>>>(
          static_cast<const __nv_bfloat16*>(x), n_rows, static_cast<const __nv_bfloat16*>(w1), b1, w2, b2, out_dim, out);
    else
      k_node_head128_mma<__half><<<grid, kNhWarps * 32, 0, stream>>>(
          static_cast<const __half*>(x), n_rows, static_cast<const __half*>(w1), b1, w2, b2, out_dim, out);
  }
  BG_LAUNCH_OK();
  return BG_OK;
}

// ------------------------------------------------------------------ EA-GNN helpers
int bg_expand_rowptr(const int32_t* rowptr, int64_t n_rows, int64_t n_entries, int32_t* row_of, int32_t* iota,
                     void* nonempty, int nonempty_dtype, int as_count, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n_rows < 0 || n_entries < 0 || (n_rows > 0 && !rowptr))
    return fail(BG_ERR_INVALID, "bg_expand_rowptr: bad argument");
  if (n_rows == 0) return BG_OK;
  const unsigned grid = grid_for(n_rows * 32, 256, sm_count() * 32);
  if (!nonempty) k_expand_rowptr<float><<<grid, 256, 0, stream>>>(rowptr, n_rows, row_of, iota, nullptr, 0);
  else if (nonempty_dtype == BG_BF16) k_expand_rowptr<__nv_bfloat16><<<grid, 256, 0, stream>>>(rowptr, n_rows, row_of, iota, static_cast<__nv_bfloat16*>(nonempty), as_count);
  else if (nonempty_dtype == BG_F16) k_expand_rowptr<__half><<<grid, 256, 0, stream>>>(rowptr, n_rows, row_of, iota, static_cast<__half*>(nonempty), as_count);
  else if (nonempty_dtype == BG_F32) k_expand_rowptr<float><<<grid, 256, 0, stream>>>(rowptr, n_rows, row_of, iota, static_cast<float*>(nonempty), as_count);
  else return fail(BG_ERR_INVALID, "bg_expand_rowptr: bad dtype");
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_add(const void* a, const void* b, const void* c, void* out, int dtype, int64_t n, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || (n > 0 && (!a || !b || !out))) return fail(BG_ERR_INVALID, "bg_add: bad argument");
  if (n == 0) return BG_OK;
  const unsigned grid = grid_for(n, 256, sm_count() * 16);
  if (dtype == BG_BF16) k_add<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(a), static_cast<const __nv_bfloat16*>(b), static_cast<const __nv_bfloat16*>(c), static_cast<__nv_bfloat16*>(out), n);
  else if (dtype == BG_F16) k_add<__half><<<grid, 256, 0, stream>>>(static_cast<const __half*>(a), static_cast<const __half*>(b), static_cast<const __half*>(c), static_cast<__half*>(out), n);
  else if (dtype == BG_F32) k_add<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(a), static_cast<const float*>(b), static_cast<const float*>(c), static_cast<float*>(out), n);
  else return fail(BG_ERR_INVALID, "bg_add: bad dtype");
  BG_LAUNCH_OK();
  return BG_OK;
}


// ------------------------------------------------------------------ training step
static inline int stat_grid(int64_t N) { return (int)min64(ceil_div64(N > 0 ? N : 1, kStatWarps), (int64_t)sm_count() * 2); }
static inline DropArgs drop_args(float p, uint64_t seed) {
  DropArgs d;
  d.seed = seed; d.thr = dropout_threshold(p); d.inv_keep = d.thr ? 1.f / (1.f - p) : 1.f;
  return d;
}
#define BG_BY_DTYPE(dtype, CALL)                                    \
  if ((dtype) == BG_BF16) { using T = __nv_bfloat16; CALL; }       \
  else if ((dtype) == BG_F16) { using T = __half; CALL; }          \
  else if ((dtype) == BG_F32) { using T = float; CALL; }           \
  else return fail(BG_ERR_INVALID, "bad dtype");

// ------------------------------------------------------------------ SAGPooling (GraphSAGE_SAG / EAGNN_SAG)
int bg_sag_workspace_bytes(int64_t N, int64_t E, int64_t G, size_t* bytes_host) {
  if (!bytes_host || N < 0 || E < 0 || G < 0) return fail(BG_ERR_INVALID, "bg_sag_workspace_bytes: bad argument");
  *bytes_host = sag_workspace_layout(nullptr, N, E, G).bytes;
  return BG_OK;
}

// The 512- and 128-wide entry points share everything but the dot pass over x (k_sag_dots<T, width>)
static int sag_select_impl(const char* fn, int width, const void* x, int dtype, int64_t N, const int32_t* rowptr,
                           const int32_t* col, const int32_t* big_rows, int32_t n_big, const float* w_l, const float* w_r,
                           float bias, float sign, const int32_t* graph_ptr, int64_t G, float ratio,
                           const int64_t* edge_index, int64_t E, float* score, int32_t* new_id, int32_t* perm,
                           int64_t* batch_out, float* score_out, int32_t* new_graph_ptr, int32_t* info, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || E < 0 || G < 0 || N >= 0x7fffffffLL || E >= 0x7fffffffLL || G >= 0x7fffffffLL || n_big < 0)
    return fail_in(BG_ERR_INVALID, fn, "sizes out of range");
  if (!(ratio > 0.f) || ratio > 1.f) return fail_in(BG_ERR_INVALID, fn, "ratio must be in (0, 1]");
  if (!info || !new_graph_ptr || !graph_ptr || !workspace) return fail_in(BG_ERR_INVALID, fn, "null pointer");
  if (N > 0 && (!x || !aligned16(x) || !rowptr || !w_l || !w_r || !score || !new_id || !perm || !batch_out || !score_out))
    return fail_in(BG_ERR_INVALID, fn, "null or misaligned pointer");
  if ((E > 0 && (!edge_index || !col)) || (n_big > 0 && !big_rows)) return fail_in(BG_ERR_INVALID, fn, "null pointer");
  SagWorkspace w = sag_workspace_layout(workspace, N, E, G);
  if (workspace_bytes < w.bytes) return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  if (width != kHidden && dtype != BG_BF16 && dtype != BG_F16 && dtype != BG_F32)
    return fail_in(BG_ERR_INVALID, fn, "bad dtype");                                    // (512: BG_BY_DTYPE)
  const int sms = sm_count();
  BG_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int32_t) * 2, stream));
  if (N > 0) {
    const unsigned grid = grid_for(N * 32, kSagWarps * 32, sms * 8);
    if (width == kHidden) {
      BG_BY_DTYPE(dtype, (k_sag_dots<T, kHidden><<<grid, kSagWarps * 32, 0, stream>>>(static_cast<const T*>(x), N, w_l, w_r, w.p, w.q)));
    } else {
      BG_BY_DTYPE(dtype, (k_sag_dots<T, kW128><<<grid, kSagWarps * 32, 0, stream>>>(static_cast<const T*>(x), N, w_l, w_r, w.p, w.q)));
    }
    BG_LAUNCH_OK();
    k_sag_score<true><<<grid_for(N * 8, 256, sms * 8), 256, 0, stream>>>(rowptr, col, w.p, w.q, bias, sign, N, score);
    BG_LAUNCH_OK();
    if (n_big > 0) {
      k_sag_score_big<true><<<(unsigned)n_big, 256, 0, stream>>>(rowptr, col, big_rows, w.p, w.q, bias, sign, score);
      BG_LAUNCH_OK();
    }
  }
  k_sag_plan<<<1, 1024, 0, stream>>>(graph_ptr, (int32_t)G, ratio, new_graph_ptr, w.tile_ptr, info);
  BG_LAUNCH_OK();
  if (N > 0 && G > 0) {
    static bool sort_attr_set = false;
    const int sort_smem = kSagSortMax * (int)sizeof(unsigned long long);
    if (!sort_attr_set) {
      BG_CUDA_OK(cudaFuncSetAttribute(k_sag_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, sort_smem));
      sort_attr_set = true;
    }
    k_sag_sort<<<(unsigned)min64(G, sms), 1024, sort_smem, stream>>>(score, graph_ptr, (int32_t)G, new_graph_ptr, new_id, perm,
                                                                     batch_out, score_out);
    BG_LAUNCH_OK();
    const unsigned tiles = (unsigned)(ceil_div64(N, kRankTileI) + G);       // >= sum_g ceil(n_g / tile)
    k_sag_rank<<<tiles, kRankThreads, 0, stream>>>(score, graph_ptr, (int32_t)G, new_graph_ptr, w.tile_ptr, new_id, perm,
                                                  batch_out, score_out);
    BG_LAUNCH_OK();
  }
  if (E > 0) {
    k_sag_edge_count<<<(unsigned)w.n_edge_blocks, 1024, 0, stream>>>(edge_index, E, N, new_id, w.block_sums);
    BG_LAUNCH_OK();
    k_sag_scan_sums<<<1, 1024, 0, stream>>>(w.block_sums, w.n_edge_blocks, info + 1);
    BG_LAUNCH_OK();
  }
  return BG_OK;
}

int bg_sag_select(const void* x, int dtype, int64_t N, const int32_t* rowptr, const int32_t* col,
                  const int32_t* big_rows, int32_t n_big, const float* w_l, const float* w_r, float bias, float sign,
                  const int32_t* graph_ptr, int64_t G, float ratio, const int64_t* edge_index, int64_t E,
                  float* score, int32_t* new_id, int32_t* perm, int64_t* batch_out, float* score_out,
                  int32_t* new_graph_ptr, int32_t* info, void* workspace, size_t workspace_bytes, void* stream_) {
  return sag_select_impl("bg_sag_select", kHidden, x, dtype, N, rowptr, col, big_rows, n_big, w_l, w_r, bias, sign,
                         graph_ptr, G, ratio, edge_index, E, score, new_id, perm, batch_out, score_out, new_graph_ptr, info,
                         workspace, workspace_bytes, stream_);
}

int bg_sag_select128(const void* x, int dtype, int64_t N, const int32_t* rowptr, const int32_t* col,
                     const int32_t* big_rows, int32_t n_big, const float* w_l, const float* w_r, float bias, float sign,
                     const int32_t* graph_ptr, int64_t G, float ratio, const int64_t* edge_index, int64_t E,
                     float* score, int32_t* new_id, int32_t* perm, int64_t* batch_out, float* score_out,
                     int32_t* new_graph_ptr, int32_t* info, void* workspace, size_t workspace_bytes, void* stream_) {
  return sag_select_impl("bg_sag_select128", kW128, x, dtype, N, rowptr, col, big_rows, n_big, w_l, w_r, bias, sign,
                         graph_ptr, G, ratio, edge_index, E, score, new_id, perm, batch_out, score_out, new_graph_ptr, info,
                         workspace, workspace_bytes, stream_);
}

int bg_sag_connect(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* new_id, int64_t E_out,
                   int64_t* edge_index_out, int32_t* kept_edge, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || E < 0 || E_out < 0 || E_out > E) return fail(BG_ERR_INVALID, "bg_sag_connect: bad size");
  if (E_out == 0) return BG_OK;
  if (!edge_index || !new_id || !edge_index_out || !workspace) return fail(BG_ERR_INVALID, "bg_sag_connect: null pointer");
  SagWorkspace w = sag_workspace_layout(workspace, N, E, 0);       // the block offsets bg_sag_select left behind
  if (workspace_bytes < w.bytes) return fail(BG_ERR_WORKSPACE, "bg_sag_connect: workspace too small");
  k_sag_edge_write<<<(unsigned)w.n_edge_blocks, 1024, 0, stream>>>(edge_index, E, N, new_id, w.block_sums, E_out,
                                                                  edge_index_out, kept_edge);
  BG_LAUNCH_OK();
  return BG_OK;
}

static int sag_pool_backward_impl(const char* fn, int width, const void* dx_pooled, const void* x, int dtype, int64_t N,
                                  int64_t N_out, const int32_t* perm, const int32_t* new_id, const float* score, float sign,
                                  const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_rows_src,
                                  int32_t n_big_src, const float* w_l, const float* w_r, void* dx, float* t, float* dpre,
                                  void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || N_out < 0 || N_out > N || n_big_src < 0) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (N == 0) return BG_OK;
  if (!x || !new_id || !score || !rowptr_src || !w_l || !w_r || !dx || !t || !dpre || !aligned16(x) || !aligned16(dx) ||
      (N_out > 0 && (!dx_pooled || !perm || !aligned16(dx_pooled))) || (n_big_src > 0 && !big_rows_src))
    return fail_in(BG_ERR_INVALID, fn, "null or misaligned pointer");
  if (width != kHidden && dtype != BG_BF16 && dtype != BG_F16 && dtype != BG_F32)
    return fail_in(BG_ERR_INVALID, fn, "bad dtype");                                    // (512: BG_BY_DTYPE)
  const int sms = sm_count();
  BG_CUDA_OK(cudaMemsetAsync(dpre, 0, sizeof(float) * (size_t)N, stream));
  if (N_out > 0) {
    const unsigned grid = grid_for(N_out * 32, kSagWarps * 32, sms * 8);
    if (width == kHidden) {
      BG_BY_DTYPE(dtype, (k_sag_bwd_rowdot<T, kHidden><<<grid, kSagWarps * 32, 0, stream>>>(
                             static_cast<const T*>(dx_pooled), static_cast<const T*>(x), perm, score, sign, N_out, dpre)));
    } else {
      BG_BY_DTYPE(dtype, (k_sag_bwd_rowdot<T, kW128><<<grid, kSagWarps * 32, 0, stream>>>(
                             static_cast<const T*>(dx_pooled), static_cast<const T*>(x), perm, score, sign, N_out, dpre)));
    }
    BG_LAUNCH_OK();
  }
  k_sag_score<false><<<grid_for(N * 8, 256, sms * 8), 256, 0, stream>>>(rowptr_src, col_src, dpre, nullptr, 0.f, 1.f, N, t);
  BG_LAUNCH_OK();
  if (n_big_src > 0) {
    k_sag_score_big<false><<<(unsigned)n_big_src, 256, 0, stream>>>(rowptr_src, col_src, big_rows_src, dpre, nullptr, 0.f, 1.f, t);
    BG_LAUNCH_OK();
  }
  const unsigned grid = grid_for(N * 32, kSagWarps * 32, sms * 8);
  if (width == kHidden) {
    BG_BY_DTYPE(dtype, (k_sag_bwd_dx<T, kHidden><<<grid, kSagWarps * 32, 0, stream>>>(
                           static_cast<const T*>(dx_pooled), new_id, score, t, dpre, w_l, w_r, N, static_cast<T*>(dx))));
  } else {
    BG_BY_DTYPE(dtype, (k_sag_bwd_dx<T, kW128><<<grid, kSagWarps * 32, 0, stream>>>(
                           static_cast<const T*>(dx_pooled), new_id, score, t, dpre, w_l, w_r, N, static_cast<T*>(dx))));
  }
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_sag_pool_backward(const void* dx_pooled, const void* x, int dtype, int64_t N, int64_t N_out, const int32_t* perm,
                         const int32_t* new_id, const float* score, float sign, const int32_t* rowptr_src,
                         const int32_t* col_src, const int32_t* big_rows_src, int32_t n_big_src, const float* w_l,
                         const float* w_r, void* dx, float* t, float* dpre, void* stream_) {
  return sag_pool_backward_impl("bg_sag_pool_backward", kHidden, dx_pooled, x, dtype, N, N_out, perm, new_id, score, sign,
                                rowptr_src, col_src, big_rows_src, n_big_src, w_l, w_r, dx, t, dpre, stream_);
}

int bg_sag_pool_backward128(const void* dx_pooled, const void* x, int dtype, int64_t N, int64_t N_out, const int32_t* perm,
                            const int32_t* new_id, const float* score, float sign, const int32_t* rowptr_src,
                            const int32_t* col_src, const int32_t* big_rows_src, int32_t n_big_src, const float* w_l,
                            const float* w_r, void* dx, float* t, float* dpre, void* stream_) {
  return sag_pool_backward_impl("bg_sag_pool_backward128", kW128, dx_pooled, x, dtype, N, N_out, perm, new_id, score, sign,
                                rowptr_src, col_src, big_rows_src, n_big_src, w_l, w_r, dx, t, dpre, stream_);
}

int bg_max_bwd_workspace_bytes(int32_t n_big_tgt, int32_t n_big_src, size_t* bytes_host) {
  if (!bytes_host || n_big_tgt < 0 || n_big_src < 0) return fail(BG_ERR_INVALID, "bg_max_bwd_workspace_bytes: bad argument");
  const int32_t m = n_big_tgt > n_big_src ? n_big_tgt : n_big_src;
  *bytes_host = (size_t)m * kMaxBwdSlices * kHidden * sizeof(float) + 256;
  return BG_OK;
}

static int max_aggregate_backward_impl(const char* fn, int width, const void* x, const void* agg, const void* dagg, int dtype,
                                       int64_t N, const int32_t* rowptr_tgt, const int32_t* col_tgt, const int32_t* big_tgt,
                                       int32_t n_big_tgt, const int32_t* rowptr_src, const int32_t* col_src,
                                       const int32_t* big_src, int32_t n_big_src, void* w_scratch, void* dx, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || n_big_tgt < 0 || n_big_src < 0) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (N == 0) return BG_OK;
  if (!x || !agg || !dagg || !rowptr_tgt || !rowptr_src || !w_scratch || !dx || !aligned16(x) || !aligned16(agg) ||
      !aligned16(dagg) || !aligned16(w_scratch) || !aligned16(dx) || (n_big_tgt > 0 && !big_tgt) || (n_big_src > 0 && !big_src))
    return fail_in(BG_ERR_INVALID, fn, "null or misaligned pointer");
  size_t need = 0;
  bg_max_bwd_workspace_bytes(n_big_tgt, n_big_src, &need);
  if ((n_big_tgt > 0 || n_big_src > 0) && (!workspace || workspace_bytes < need))
    return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  if (width != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  const unsigned grid = grid_for(N * 32, kMaxBwdWarps * 32, sm_count() * 8);
  if (width == kHidden) {
    BG_BY_DTYPE(dtype, (launch_max_bwd<T, kHidden>(x, agg, dagg, N, rowptr_tgt, col_tgt, big_tgt, n_big_tgt, rowptr_src, col_src,
                                                   big_src, n_big_src, w_scratch, dx, static_cast<float*>(workspace), grid, stream)));
  } else {
    BG_BY_DTYPE(dtype, (launch_max_bwd<T, kW128>(x, agg, dagg, N, rowptr_tgt, col_tgt, big_tgt, n_big_tgt, rowptr_src, col_src,
                                                 big_src, n_big_src, w_scratch, dx, static_cast<float*>(workspace), grid, stream)));
  }
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_max_aggregate_backward(const void* x, const void* agg, const void* dagg, int dtype, int64_t N,
                              const int32_t* rowptr_tgt, const int32_t* col_tgt, const int32_t* big_tgt, int32_t n_big_tgt,
                              const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_src, int32_t n_big_src,
                              void* w_scratch, void* dx, void* workspace, size_t workspace_bytes, void* stream_) {
  return max_aggregate_backward_impl("bg_max_aggregate_backward", kHidden, x, agg, dagg, dtype, N, rowptr_tgt, col_tgt, big_tgt,
                                     n_big_tgt, rowptr_src, col_src, big_src, n_big_src, w_scratch, dx, workspace,
                                     workspace_bytes, stream_);
}

int bg_max_aggregate_backward128(const void* x, const void* agg, const void* dagg, int dtype, int64_t N,
                                 const int32_t* rowptr_tgt, const int32_t* col_tgt, const int32_t* big_tgt, int32_t n_big_tgt,
                                 const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_src, int32_t n_big_src,
                                 void* w_scratch, void* dx, void* workspace, size_t workspace_bytes, void* stream_) {
  return max_aggregate_backward_impl("bg_max_aggregate_backward128", kW128, x, agg, dagg, dtype, N, rowptr_tgt, col_tgt,
                                     big_tgt, n_big_tgt, rowptr_src, col_src, big_src, n_big_src, w_scratch, dx, workspace,
                                     workspace_bytes, stream_);
}

static int gather_rows_impl(const char* fn, int width, const void* x, int dtype, int64_t ldx, const int32_t* row_index,
                            const float* row_scale, int64_t n_rows_out, void* out, int64_t ldo, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n_rows_out < 0 || ldx < width || ldo < width) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (n_rows_out == 0) return BG_OK;
  if (!x || !out || !row_index || !aligned16(x) || !aligned16(out)) return fail_in(BG_ERR_INVALID, fn, "null or misaligned pointer");
  const int esz = (dtype == BG_F32) ? 4 : 2;
  if ((ldx * esz) % 16 != 0 || (ldo * esz) % 16 != 0) return fail_in(BG_ERR_INVALID, fn, "rows must be 16-byte aligned");
  if (width != kHidden && dtype != BG_BF16 && dtype != BG_F16 && dtype != BG_F32)
    return fail_in(BG_ERR_INVALID, fn, "bad dtype");                                    // (512: BG_BY_DTYPE)
  const unsigned grid = grid_for(n_rows_out * 32, kSagWarps * 32, sm_count() * 8);
  if (width == kHidden) {
    BG_BY_DTYPE(dtype, (k_gather_rows<T, kHidden><<<grid, kSagWarps * 32, 0, stream>>>(
                           static_cast<const T*>(x), ldx, row_index, row_scale, n_rows_out, static_cast<T*>(out), ldo)));
  } else {
    BG_BY_DTYPE(dtype, (k_gather_rows<T, kW128><<<grid, kSagWarps * 32, 0, stream>>>(
                           static_cast<const T*>(x), ldx, row_index, row_scale, n_rows_out, static_cast<T*>(out), ldo)));
  }
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_gather_rows(const void* x, int dtype, int64_t ldx, const int32_t* row_index, const float* row_scale,
                   int64_t n_rows_out, void* out, int64_t ldo, void* stream_) {
  return gather_rows_impl("bg_gather_rows", kHidden, x, dtype, ldx, row_index, row_scale, n_rows_out, out, ldo, stream_);
}

int bg_gather_rows128(const void* x, int dtype, int64_t ldx, const int32_t* row_index, const float* row_scale,
                      int64_t n_rows_out, void* out, int64_t ldo, void* stream_) {
  return gather_rows_impl("bg_gather_rows128", kW128, x, dtype, ldx, row_index, row_scale, n_rows_out, out, ldo, stream_);
}

int bg_index_invert(const int32_t* perm, int64_t n, int32_t* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || (n > 0 && (!perm || !out))) return fail(BG_ERR_INVALID, "bg_index_invert: bad argument");
  if (n == 0) return BG_OK;
  k_index_invert<<<grid_for(n, 256, sm_count() * 16), 256, 0, stream>>>(perm, n, out);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_index_gather(const int32_t* table, const int32_t* idx, int64_t n, int32_t* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || (n > 0 && (!table || !idx || !out))) return fail(BG_ERR_INVALID, "bg_index_gather: bad argument");
  if (n == 0) return BG_OK;
  k_index_gather<<<grid_for(n, 256, sm_count() * 16), 256, 0, stream>>>(table, idx, n, out);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_train_workspace_bytes(int64_t N, size_t* bytes_host) {
  if (!bytes_host || N < 0) return fail(BG_ERR_INVALID, "bg_train_workspace_bytes: bad argument");
  *bytes_host = (size_t)stat_grid(N) * 2 * kHidden * sizeof(float) + 2 * kHidden * sizeof(float) + 256;
  return BG_OK;
}

extern "C++" {
template <int kW>
static int bn_batch_stats_impl(const char* fn, const void* u, int dtype, int64_t N, const float* gamma, const float* beta,
                               float eps, float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                               float* a_out, float* shift_out, float* mean_out, float* invstd_out,
                               void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N <= 0) return fail_in(BG_ERR_INVALID, fn, "needs at least one row");
  if (!u || !aligned16(u) || !gamma || !beta || !a_out || !shift_out || !mean_out || !invstd_out)
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  if ((running_mean != nullptr) != (running_var != nullptr)) return fail_in(BG_ERR_INVALID, fn, "running_mean and running_var go together");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  size_t need = 0;
  bg_train_workspace_bytes(N, &need);
  if (!workspace || workspace_bytes < need) return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  float* partial = static_cast<float*>(workspace);
  const int grid = stat_grid(N);
  const DropArgs nodrop = drop_args(0.f, 0);
  BG_BY_DTYPE(dtype, (k_col_stats<T, 0, kW><<<grid, kStatWarps * 32, 0, stream>>>(static_cast<const T*>(u), nullptr, nullptr, N,
                                                                              nullptr, nullptr, nodrop, partial)))
  BG_LAUNCH_OK();
  BnVectors out{a_out, shift_out, mean_out, invstd_out};
  k_bn_fwd_finalize<kW><<<kW / 64, kHidden, 0, stream>>>(partial, grid, N, gamma, beta, eps, momentum, running_mean, running_var,
                                                        reinterpret_cast<long long*>(num_batches_tracked), out);
  BG_LAUNCH_OK();
  return BG_OK;
}
}  // extern "C++"

int bg_bn_batch_stats(const void* u, int dtype, int64_t N, const float* gamma, const float* beta, float eps,
                      float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                      float* a_out, float* shift_out, float* mean_out, float* invstd_out,
                      void* workspace, size_t workspace_bytes, void* stream_) {
  return bn_batch_stats_impl<kHidden>("bg_bn_batch_stats", u, dtype, N, gamma, beta, eps, momentum, running_mean, running_var,
                                      num_batches_tracked, a_out, shift_out, mean_out, invstd_out, workspace, workspace_bytes, stream_);
}

int bg_bn_batch_stats128(const void* u, int dtype, int64_t N, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                         float* a_out, float* shift_out, float* mean_out, float* invstd_out,
                         void* workspace, size_t workspace_bytes, void* stream_) {
  return bn_batch_stats_impl<kW128>("bg_bn_batch_stats128", u, dtype, N, gamma, beta, eps, momentum, running_mean, running_var,
                                    num_batches_tracked, a_out, shift_out, mean_out, invstd_out, workspace, workspace_bytes, stream_);
}

extern "C++" {
template <int kW>
static int bn_act_forward_impl(const char* fn, const void* u, const void* x_prev, void* y, int dtype, int64_t N, const float* a,
                               const float* shift, float dropout_p, uint64_t seed, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || !(dropout_p >= 0.f && dropout_p < 1.f)) return fail_in(BG_ERR_INVALID, fn, "bad size / dropout_p");
  if (N == 0) return BG_OK;
  if (!u || !y || !a || !shift || !aligned16(u) || !aligned16(y) || (x_prev && !aligned16(x_prev)))
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  const unsigned grid = grid_for(N * 32, 256, sm_count() * 8);
  const DropArgs d = drop_args(dropout_p, seed);
  BG_BY_DTYPE(dtype, (k_bn_act_fwd<T, kW><<<grid, 256, 0, stream>>>(static_cast<const T*>(u), static_cast<const T*>(x_prev),
                                                                    static_cast<T*>(y), N, a, shift, d)))
  BG_LAUNCH_OK();
  return BG_OK;
}
}  // extern "C++"

int bg_bn_act_forward(const void* u, const void* x_prev, void* y, int dtype, int64_t N, const float* a,
                      const float* shift, float dropout_p, uint64_t seed, void* stream_) {
  return bn_act_forward_impl<kHidden>("bg_bn_act_forward", u, x_prev, y, dtype, N, a, shift, dropout_p, seed, stream_);
}

int bg_bn_act_forward128(const void* u, const void* x_prev, void* y, int dtype, int64_t N, const float* a,
                         const float* shift, float dropout_p, uint64_t seed, void* stream_) {
  return bn_act_forward_impl<kW128>("bg_bn_act_forward128", u, x_prev, y, dtype, N, a, shift, dropout_p, seed, stream_);
}

extern "C++" {
template <int kW>
static int sage_backward_rows_impl(const char* fn, const void* u, const void* dy, const void* dy2, const float* inv_norm,
                                   const int32_t* rowptr, int dtype, int64_t N, const float* a, const float* shift,
                                   const float* mean, const float* invstd, float dropout_p, uint64_t seed, float* dgamma,
                                   float* dbeta, int accumulate, void* dz, void* dz_scaled, void* g_out,
                                   void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N <= 0) return fail_in(BG_ERR_INVALID, fn, "needs at least one row");
  if (!(dropout_p >= 0.f && dropout_p < 1.f)) return fail_in(BG_ERR_INVALID, fn, "bad dropout_p");
  if (!u || !dy || !dz || !a || !shift || !aligned16(u) || !aligned16(dy) || !aligned16(dz) || (dy2 && !aligned16(dy2)) ||
      (dz_scaled && (!aligned16(dz_scaled) || !rowptr)) || (g_out && !aligned16(g_out)))
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  const bool bn = mean != nullptr;
  if (bn && (!invstd || !dgamma || !dbeta)) return fail_in(BG_ERR_INVALID, fn, "BatchNorm needs mean, invstd, dgamma, dbeta");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  size_t need = 0;
  bg_train_workspace_bytes(N, &need);
  if (!workspace || workspace_bytes < need) return fail_in(BG_ERR_WORKSPACE, fn, "workspace too small");
  float* partial = static_cast<float*>(workspace);
  const int grid = stat_grid(N);
  float* k0 = partial + (size_t)grid * 2 * kW;
  float* k1 = k0 + kW;
  const DropArgs d = drop_args(dropout_p, seed);
  if (bn) {
    BG_BY_DTYPE(dtype, (k_col_stats<T, 1, kW><<<grid, kStatWarps * 32, 0, stream>>>(static_cast<const T*>(u), static_cast<const T*>(dy),
                                                                                static_cast<const T*>(dy2), N, a, shift, d, partial)))
    BG_LAUNCH_OK();
    BnVectors v{const_cast<float*>(a), const_cast<float*>(shift), const_cast<float*>(mean), const_cast<float*>(invstd)};
    k_bn_bwd_finalize<kW><<<kW / 64, kHidden, 0, stream>>>(partial, grid, N, v, dgamma, dbeta, accumulate, k0, k1);
    BG_LAUNCH_OK();
  } else {
    BG_CUDA_OK(cudaMemsetAsync(k0, 0, 2 * kW * sizeof(float), stream));
  }
  const unsigned rgrid = grid_for(N * 32, 256, sm_count() * 8);
  BG_BY_DTYPE(dtype, (k_sage_bwd_rows<T, kW><<<rgrid, 256, 0, stream>>>(static_cast<const T*>(u), static_cast<const T*>(dy),
                                                                        static_cast<const T*>(dy2), N, inv_norm, rowptr, a, shift, k0, k1, d,
                                                                        static_cast<T*>(dz), static_cast<T*>(dz_scaled), static_cast<T*>(g_out))))
  BG_LAUNCH_OK();
  return BG_OK;
}
}  // extern "C++"

int bg_sage_backward_rows(const void* u, const void* dy, const void* dy2, const float* inv_norm, const int32_t* rowptr,
                          int dtype, int64_t N, const float* a, const float* shift, const float* mean,
                          const float* invstd, float dropout_p, uint64_t seed, float* dgamma, float* dbeta,
                          int accumulate, void* dz, void* dz_scaled, void* g_out,
                          void* workspace, size_t workspace_bytes, void* stream_) {
  return sage_backward_rows_impl<kHidden>("bg_sage_backward_rows", u, dy, dy2, inv_norm, rowptr, dtype, N, a, shift, mean, invstd,
                                          dropout_p, seed, dgamma, dbeta, accumulate, dz, dz_scaled, g_out, workspace,
                                          workspace_bytes, stream_);
}

int bg_sage_backward_rows128(const void* u, const void* dy, const void* dy2, const float* inv_norm, const int32_t* rowptr,
                             int dtype, int64_t N, const float* a, const float* shift, const float* mean,
                             const float* invstd, float dropout_p, uint64_t seed, float* dgamma, float* dbeta,
                             int accumulate, void* dz, void* dz_scaled, void* g_out,
                             void* workspace, size_t workspace_bytes, void* stream_) {
  return sage_backward_rows_impl<kW128>("bg_sage_backward_rows128", u, dy, dy2, inv_norm, rowptr, dtype, N, a, shift, mean,
                                        invstd, dropout_p, seed, dgamma, dbeta, accumulate, dz, dz_scaled, g_out, workspace,
                                        workspace_bytes, stream_);
}

int bg_transpose_chunks(const void* in, int dtype, int64_t n_rows, int32_t n_cols, int64_t ld, int32_t n_chunks,
                        int64_t chunk_k, int32_t out_rows_per_chunk, void* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (out_rows_per_chunk <= 0) out_rows_per_chunk = n_cols;
  if (n_rows < 0 || n_cols <= 0 || n_cols % 32 != 0 || n_chunks <= 0 || chunk_k <= 0 || chunk_k % 32 != 0 ||
      (int64_t)n_chunks * chunk_k < n_rows || ld < n_cols || out_rows_per_chunk < n_cols)
    return fail(BG_ERR_INVALID, "bg_transpose_chunks: bad shape (n_cols, chunk_k multiples of 32; n_chunks*chunk_k >= n_rows)");
  if (!in || !out) return fail(BG_ERR_INVALID, "bg_transpose_chunks: bad pointer");
  dim3 grid((unsigned)((int64_t)n_chunks * chunk_k / 32), (unsigned)(n_cols / 32)), block(32, 8);
  BG_BY_DTYPE(dtype, (k_transpose_chunks<T><<<grid, block, 0, stream>>>(static_cast<const T*>(in), n_rows, n_cols, ld, chunk_k, out_rows_per_chunk, static_cast<T*>(out))))
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_mask_narrow(const void* in, int in_dtype, int64_t ld_in, const void* mask, int mask_dtype, int64_t ld_mask,
                   int64_t M, int32_t n_cols, float* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (M < 0 || n_cols <= 0 || ld_in < n_cols || (mask && ld_mask < n_cols)) return fail(BG_ERR_INVALID, "bg_mask_narrow: bad shape");
  if (umma_format_of(in_dtype) < 0 || (mask && umma_format_of(mask_dtype) < 0)) return fail(BG_ERR_INVALID, "bg_mask_narrow: bad dtype");
  if (M == 0) return BG_OK;
  if (!in || !out) return fail(BG_ERR_INVALID, "bg_mask_narrow: bad pointer");
  k_mask_narrow<<<grid_for(M * n_cols, 256, sm_count() * 8), 256, 0, stream>>>(in, in_dtype, ld_in, mask, mask_dtype, ld_mask, M, n_cols, out);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_reduce_partials(const float* partial, int32_t n_chunks, int64_t n, float* out, int accumulate, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || n_chunks <= 0 || (n > 0 && (!partial || !out))) return fail(BG_ERR_INVALID, "bg_reduce_partials: bad argument");
  if (n == 0) return BG_OK;
  k_reduce_partials<<<grid_for(n, 256, sm_count() * 8), 256, 0, stream>>>(partial, n_chunks, n, out, accumulate);
  BG_LAUNCH_OK();
  return BG_OK;
}

static inline int colsum_chunks(int64_t rows) { return (int)min64(ceil_div64(rows > 0 ? rows : 1, 64), 128); }
int bg_colsum_workspace_bytes(int64_t rows, int32_t cols, size_t* bytes_host) {
  if (!bytes_host || rows < 0 || cols <= 0) return fail(BG_ERR_INVALID, "bg_colsum_workspace_bytes: bad argument");
  *bytes_host = (size_t)colsum_chunks(rows) * cols * sizeof(float) + 256;
  return BG_OK;
}
int bg_colsum(const void* in, int dtype, int64_t rows, int32_t cols, int64_t ld, float* out, int accumulate,
              void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (rows < 0 || cols <= 0 || ld < cols || !out) return fail(BG_ERR_INVALID, "bg_colsum: bad argument");
  if (umma_format_of(dtype) < 0) return fail(BG_ERR_INVALID, "bg_colsum: bad dtype");
  if (rows == 0) { if (!accumulate) BG_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * cols, stream)); return BG_OK; }
  size_t need = 0;
  bg_colsum_workspace_bytes(rows, cols, &need);
  if (!in || !workspace || workspace_bytes < need) return fail(BG_ERR_WORKSPACE, "bg_colsum: workspace too small");
  const int chunks = colsum_chunks(rows);
  float* partial = static_cast<float*>(workspace);
  k_colsum_partial<<<dim3((unsigned)ceil_div64(cols, 32), (unsigned)chunks), dim3(32, 8), 0, stream>>>(in, dtype, rows, cols, ld, partial);
  BG_LAUNCH_OK();
  k_reduce_partials<<<grid_for(cols, 256, 8), 256, 0, stream>>>(partial, chunks, cols, out, accumulate);
  BG_LAUNCH_OK();
  return BG_OK;
}

extern "C++" {
template <int kW>
static int pool_backward_impl(const char* fn, const float* dpooled, int64_t ldp, const int32_t* graph_ptr, int64_t G, int pool_mode,
                              int64_t N, void* dx, int dtype, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || G <= 0 || G >= 0x7fffffffLL || ldp < kW) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (pool_mode < BG_POOL_MEAN || pool_mode > BG_POOL_SUPERNODE_WITH_POOLING) return fail_in(BG_ERR_INVALID, fn, "bad pool_mode");
  if (pool_mode == BG_POOL_SUPERNODE_WITH_POOLING && ldp < 2 * kW)
    return fail_in(BG_ERR_INVALID, fn, kW == kHidden ? "the concatenated pooling needs dpooled [G, 1024]"
                                                     : "the concatenated pooling needs dpooled [G, 256]");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  if (N == 0) return BG_OK;
  if (!dpooled || !graph_ptr || !dx || !aligned16(dx)) return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  const unsigned grid = grid_for(N * 32, 256, sm_count() * 8);
  BG_BY_DTYPE(dtype, (k_pool_bwd<T, kW><<<grid, 256, 0, stream>>>(dpooled, ldp, graph_ptr, (int)G, pool_mode, N, static_cast<T*>(dx))))
  BG_LAUNCH_OK();
  return BG_OK;
}
}  // extern "C++"

int bg_pool_backward(const float* dpooled, int64_t ldp, const int32_t* graph_ptr, int64_t G, int pool_mode, int64_t N,
                     void* dx, int dtype, void* stream_) {
  return pool_backward_impl<kHidden>("bg_pool_backward", dpooled, ldp, graph_ptr, G, pool_mode, N, dx, dtype, stream_);
}

int bg_pool_backward128(const float* dpooled, int64_t ldp, const int32_t* graph_ptr, int64_t G, int pool_mode, int64_t N,
                        void* dx, int dtype, void* stream_) {
  return pool_backward_impl<kW128>("bg_pool_backward128", dpooled, ldp, graph_ptr, G, pool_mode, N, dx, dtype, stream_);
}

static inline int sgemm_splits(int64_t M, int64_t N, int64_t K) {
  const int64_t tiles = ceil_div64(M, kSgTile) * ceil_div64(N, kSgTile);
  int64_t s = ceil_div64((int64_t)sm_count() * 2, tiles);
  const int64_t max_s = ceil_div64(K, 256);                 // at least 256 of K per split
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 512) s = 512;
  return (int)s;
}
int bg_sgemm_workspace_bytes(int64_t M, int64_t N, int64_t K, size_t* bytes_host) {
  if (!bytes_host || M < 0 || N < 0 || K < 0) return fail(BG_ERR_INVALID, "bg_sgemm_workspace_bytes: bad argument");
  *bytes_host = (size_t)sgemm_splits(M, N, K) * (size_t)M * (size_t)N * sizeof(float) + 256;
  return BG_OK;
}
int bg_sgemm(const void* a, int a_dtype, int64_t sam, int64_t sak, const void* b, int b_dtype, int64_t sbk, int64_t sbn,
             int64_t M, int64_t N, int64_t K, const float* bias, int relu, const void* mask, int mask_dtype,
             int64_t mask_ld, void* out, int out_dtype, int64_t ldo, int accumulate,
             void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (M < 0 || N < 0 || K < 0 || M >= 0x7fffffffLL || N > 65535LL * kSgTile) return fail(BG_ERR_INVALID, "bg_sgemm: bad size");
  if (umma_format_of(a_dtype) < 0 || umma_format_of(b_dtype) < 0 || umma_format_of(out_dtype) < 0 ||
      (mask && umma_format_of(mask_dtype) < 0))
    return fail(BG_ERR_INVALID, "bg_sgemm: bad dtype");
  if (M == 0 || N == 0) return BG_OK;
  if ((K > 0 && (!a || !b)) || !out || ldo < N) return fail(BG_ERR_INVALID, "bg_sgemm: bad pointer / ldo");
  size_t need = 0;
  bg_sgemm_workspace_bytes(M, N, K, &need);
  if (!workspace || workspace_bytes < need) return fail(BG_ERR_WORKSPACE, "bg_sgemm: workspace too small");
  const int splits = sgemm_splits(M, N, K);
  const int64_t k_per = ceil_div64(ceil_div64(K > 0 ? K : 1, splits), kSgK) * kSgK;
  SgemmArgs g{a, b, a_dtype, b_dtype, sam, sak, sbk, sbn, M, N, K, k_per, static_cast<float*>(workspace)};
  if (ceil_div64(M, kSgTile) > 65535) return fail(BG_ERR_UNSUPPORTED, "bg_sgemm: M too large for the grid");
  k_sgemm<<<dim3((unsigned)ceil_div64(N, kSgTile), (unsigned)ceil_div64(M, kSgTile), (unsigned)splits), 256, 0, stream>>>(g);
  BG_LAUNCH_OK();
  SgemmEpilogue e{static_cast<const float*>(workspace), splits, M, N, bias, relu, mask, mask_dtype, mask_ld, out, out_dtype, ldo, accumulate};
  k_sgemm_epilogue<<<grid_for(M * N, 256, sm_count() * 8), 256, 0, stream>>>(e);
  BG_LAUNCH_OK();
  return BG_OK;
}

extern "C++" {
template <int kW>
static int dropout_residual_impl(const char* fn, const void* x, const void* x_prev, void* y, int dtype, int64_t N,
                                 float dropout_p, uint64_t seed, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || !(dropout_p >= 0.f && dropout_p < 1.f)) return fail_in(BG_ERR_INVALID, fn, "bad size / dropout_p");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  if (N == 0) return BG_OK;
  if (!x || !y || !aligned16(x) || !aligned16(y) || (x_prev && !aligned16(x_prev))) return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  const DropArgs d = drop_args(dropout_p, seed);
  const unsigned grid = grid_for(N * 32, 256, sm_count() * 8);
  BG_BY_DTYPE(dtype, (k_dropout_residual<T, kW><<<grid, 256, 0, stream>>>(static_cast<const T*>(x), static_cast<const T*>(x_prev),
                                                                          static_cast<T*>(y), N, d)))
  BG_LAUNCH_OK();
  return BG_OK;
}

template <int kW>
static int grad_mask_impl(const char* fn, const void* dy, const void* dy2, const void* act, void* out, int dtype, int64_t N,
                          float dropout_p, uint64_t seed, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (N < 0 || !(dropout_p >= 0.f && dropout_p < 1.f)) return fail_in(BG_ERR_INVALID, fn, "bad size / dropout_p");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  if (N == 0) return BG_OK;
  if (!dy || !out || !aligned16(dy) || !aligned16(out) || (dy2 && !aligned16(dy2)) || (act && !aligned16(act)))
    return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  const DropArgs d = drop_args(dropout_p, seed);
  const unsigned grid = grid_for(N * 32, 256, sm_count() * 8);
  BG_BY_DTYPE(dtype, (k_grad_mask<T, kW><<<grid, 256, 0, stream>>>(static_cast<const T*>(dy), static_cast<const T*>(dy2),
                                                                   static_cast<const T*>(act), static_cast<T*>(out), N, d)))
  BG_LAUNCH_OK();
  return BG_OK;
}

template <int kW>
static int segment_expand_impl(const char* fn, const void* src, const int32_t* rowptr, int64_t n_rows, int mean, void* out,
                               int dtype, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n_rows < 0) return fail_in(BG_ERR_INVALID, fn, "bad size");
  if (kW != kHidden && umma_format_of(dtype) < 0) return fail_in(BG_ERR_INVALID, fn, "bad dtype");   // (512: BG_BY_DTYPE)
  if (n_rows == 0) return BG_OK;
  if (!src || !rowptr || !out || !aligned16(src) || !aligned16(out)) return fail_in(BG_ERR_INVALID, fn, "bad pointer");
  const unsigned grid = grid_for(n_rows * 32, 256, sm_count() * 8);
  BG_BY_DTYPE(dtype, (k_segment_expand<T, kW><<<grid, 256, 0, stream>>>(static_cast<const T*>(src), rowptr, n_rows, mean,
                                                                        static_cast<T*>(out))))
  BG_LAUNCH_OK();
  return BG_OK;
}
}  // extern "C++"

int bg_dropout_residual(const void* x, const void* x_prev, void* y, int dtype, int64_t N, float dropout_p, uint64_t seed, void* stream_) {
  return dropout_residual_impl<kHidden>("bg_dropout_residual", x, x_prev, y, dtype, N, dropout_p, seed, stream_);
}

int bg_dropout_residual128(const void* x, const void* x_prev, void* y, int dtype, int64_t N, float dropout_p, uint64_t seed,
                           void* stream_) {
  return dropout_residual_impl<kW128>("bg_dropout_residual128", x, x_prev, y, dtype, N, dropout_p, seed, stream_);
}

int bg_grad_mask(const void* dy, const void* dy2, const void* act, void* out, int dtype, int64_t N, float dropout_p,
                 uint64_t seed, void* stream_) {
  return grad_mask_impl<kHidden>("bg_grad_mask", dy, dy2, act, out, dtype, N, dropout_p, seed, stream_);
}

int bg_grad_mask128(const void* dy, const void* dy2, const void* act, void* out, int dtype, int64_t N, float dropout_p,
                    uint64_t seed, void* stream_) {
  return grad_mask_impl<kW128>("bg_grad_mask128", dy, dy2, act, out, dtype, N, dropout_p, seed, stream_);
}

int bg_segment_expand(const void* src, const int32_t* rowptr, int64_t n_rows, int mean, void* out, int dtype, void* stream_) {
  return segment_expand_impl<kHidden>("bg_segment_expand", src, rowptr, n_rows, mean, out, dtype, stream_);
}

int bg_segment_expand128(const void* src, const int32_t* rowptr, int64_t n_rows, int mean, void* out, int dtype, void* stream_) {
  return segment_expand_impl<kW128>("bg_segment_expand128", src, rowptr, n_rows, mean, out, dtype, stream_);
}

int bg_collate_ptr(const int64_t* sel, int64_t G, const int64_t* node_ptr, const int64_t* edge_ptr,
                   int64_t* out_node_ptr, int64_t* out_edge_ptr, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G < 0 || !out_node_ptr || !out_edge_ptr || (G > 0 && (!sel || !node_ptr || !edge_ptr)))
    return fail(BG_ERR_INVALID, "bg_collate_ptr: bad argument");
  k_collate_ptr<<<1, 1024, 0, stream>>>(sel, G, node_ptr, edge_ptr, out_node_ptr, out_edge_ptr);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_collate(const float* x_all, int32_t F, const int64_t* ei_all, int64_t E_all, const float* ea_all, int32_t Fe,
               const float* y_all, const int64_t* sel, int64_t G, const int64_t* node_ptr, const int64_t* edge_ptr,
               const int64_t* out_node_ptr, const int64_t* out_edge_ptr, int64_t n_out, int64_t e_out,
               float* x, int64_t* edge_index, float* edge_attr, int64_t* batch, float* y, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G <= 0 || F <= 0 || Fe < 0 || n_out < 0 || e_out < 0 || E_all < 0) return fail(BG_ERR_INVALID, "bg_collate: bad size");
  if (!sel || !node_ptr || !edge_ptr || !out_node_ptr || !out_edge_ptr || (n_out > 0 && (!x_all || !x || !batch)) ||
      (e_out > 0 && (!ei_all || !edge_index || (Fe > 0 && (!ea_all || !edge_attr)))))
    return fail(BG_ERR_INVALID, "bg_collate: bad pointer");
  const int sms = sm_count();
  if (n_out > 0) {
    k_collate_nodes<<<grid_for(n_out * F, 256, sms * 16), 256, 0, stream>>>(x_all, F, sel, G, node_ptr, out_node_ptr, x, batch);
    BG_LAUNCH_OK();
  }
  if (e_out > 0) {
    k_collate_edges<<<grid_for(e_out, 256, sms * 16), 256, 0, stream>>>(ei_all, E_all, ea_all, Fe, sel, G, edge_ptr, out_node_ptr,
                                                                      out_edge_ptr, edge_index, edge_attr);
    BG_LAUNCH_OK();
  }
  if (y_all && y) {
    k_collate_y<<<(unsigned)ceil_div64(G, 256), 256, 0, stream>>>(y_all, sel, G, y);
    BG_LAUNCH_OK();
  }
  return BG_OK;
}

int bg_expand_wire(const int32_t* wire_edges, int64_t E_wire, const int64_t* node_ptr, const int64_t* wire_ptr,
                   const int64_t* full_ptr, int64_t G, int64_t E_full, int64_t* edge_index, int64_t* batch, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G < 0 || E_wire < 0 || E_full < E_wire || (G > 0 && (!node_ptr || !wire_ptr || !full_ptr || !batch)) ||
      (E_full > 0 && !edge_index) || (E_wire > 0 && !wire_edges))
    return fail(BG_ERR_INVALID, "bg_expand_wire: bad argument");
  if (G == 0) return BG_OK;
  k_expand_wire<<<(unsigned)min64(G, (int64_t)sm_count() * 8), 256, 0, stream>>>(wire_edges, E_wire, node_ptr, wire_ptr, full_ptr, G,
                                                                               E_full, edge_index, batch);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_eigen_loss(const float* pred, const float* y, int64_t G, float scale, float center, float eps,
                  float* out2, float* dpred, float* accum3, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (G <= 0 || !pred || !y || !out2) return fail(BG_ERR_INVALID, "bg_eigen_loss: bad argument");
  k_eigen_loss<<<1, 256, 0, stream>>>(pred, y, G, scale, center, eps, out2, dpred, accum3);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_dropout_mask(uint64_t seed, float dropout_p, int64_t n_rows, uint8_t* keep, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n_rows < 0 || (n_rows > 0 && !keep) || !(dropout_p >= 0.f && dropout_p < 1.f)) return fail(BG_ERR_INVALID, "bg_dropout_mask: bad argument");
  if (n_rows == 0) return BG_OK;
  k_dropout_mask<<<grid_for(n_rows * kHidden, 256, sm_count() * 8), 256, 0, stream>>>(seed, dropout_threshold(dropout_p), n_rows, keep);
  BG_LAUNCH_OK();
  return BG_OK;
}

// ------------------------------------------------------------------ helpers
int bg_cast_f32(const float* src, void* dst, int dst_dtype, int64_t n, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || (n > 0 && (!src || !dst))) return fail(BG_ERR_INVALID, "bg_cast_f32: bad argument");
  if (dst_dtype != BG_BF16 && dst_dtype != BG_F16) return fail(BG_ERR_INVALID, "bg_cast_f32: dst_dtype must be bf16 or f16");
  if (n == 0) return BG_OK;
  const unsigned grid = grid_for(n, 256, sm_count() * 8);
  if (dst_dtype == BG_BF16) k_cast_f32_16<__nv_bfloat16><<<grid, 256, 0, stream>>>(src, static_cast<__nv_bfloat16*>(dst), n);
  else k_cast_f32_16<__half><<<grid, 256, 0, stream>>>(src, static_cast<__half*>(dst), n);
  BG_LAUNCH_OK();
  return BG_OK;
}

int bg_split_tf32(const float* src, float* hi, float* lo, int64_t n, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (n < 0 || (n > 0 && (!src || !lo))) return fail(BG_ERR_INVALID, "bg_split_tf32: bad argument");
  if (n == 0) return BG_OK;
  k_split_tf32<<<grid_for(n, 256, sm_count() * 8), 256, 0, stream>>>(src, hi, lo, n);
  BG_LAUNCH_OK();
  return BG_OK;
}

}  // extern "C"
