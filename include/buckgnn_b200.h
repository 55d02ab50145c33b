/* buckgnn_b200 -- C ABI of the B200-native BuckGNN forward hot path.
 *
 * The reference (omerkurt-okt/buck-gnn) is pure Python: its hot path,
 * `BuckGNN.forward` (Models/BuckGNN.py:311-526), bottoms out in torch_geometric /
 * torch_scatter library kernels.  It has no FFI of its own, so the boundary a
 * maintainer binds is the set of operators that forward calls; each entry point
 * below names the reference call site it replaces.  The Python host
 * (buckgnn_b200/capi.py, ctypes) is the only caller; INTEGRATION.md shows the
 * binding.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *    buffers are borrowed for the duration of the call, never retained;
 *  - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *    all work is enqueued on it, nothing synchronises unless stated;
 *  - return value: BG_OK (0) or a negative bg_status; bg_last_error() gives the
 *    text of the last failure on the calling thread.  Nothing throws;
 *  - no allocation happens inside: workspace sizes are queried first so the host
 *    framework (torch's caching allocator) owns all memory;
 *  - matrices are row-major; `ld*` are leading dimensions in ELEMENTS.
 *  - the library is compiled for sm_100a only; bg_device_check() says whether the
 *    current device can run it.  There is no CPU fallback.
 */
#ifndef BUCKGNN_B200_H_
#define BUCKGNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BG_ABI_VERSION 11

typedef enum bg_status {
  BG_OK = 0,
  BG_ERR_INVALID = -1,      /* bad argument (null pointer, size, alignment, enum) */
  BG_ERR_CUDA = -2,         /* a CUDA runtime/driver call failed; see bg_last_error() */
  BG_ERR_WORKSPACE = -3,    /* workspace too small */
  BG_ERR_UNSUPPORTED = -4,  /* shape / mode outside what the kernels are built for */
  BG_ERR_DEVICE = -5        /* current device is not sm_100 */
} bg_status;

typedef enum bg_dtype { BG_BF16 = 0, BG_F32 = 1, BG_F16 = 2 } bg_dtype;

/* SAGEConv(aggr=...) values used by the reference (Models/BuckGNN.py:118,130,145,160,175);
 * 'add' and 'sum' are the same reduction. */
typedef enum bg_aggr { BG_AGGR_MEAN = 0, BG_AGGR_SUM = 1, BG_AGGR_MAX = 2 } bg_aggr;

int bg_abi_version(void);
const char* bg_last_error(void);
/* BG_OK if the current CUDA device is compute capability 10.x */
int bg_device_check(void);
/* info about the last barrier watchdog trip (debugging aid): 4 words copied to host */
int bg_watchdog_info_host(uint32_t* out4_host);
/* SM partition for kernels that are meant to run side by side on two streams: bg_gemm512 launches at most
 * `gemm_sms` CTAs (rounded down to CTA pairs) and bg_sage_aggregate at most `agg_sms`; 0 = the whole device.
 * Process-wide, takes effect at the next launch. */
int bg_set_sm_partition(int gemm_sms, int agg_sms);

/* ------------------------------------------------------------------ K1: CSR build
 * Replaces the implicit gather/scatter indexing inside PyG's
 * `SAGEConv.propagate` (called at Models/BuckGNN.py:342,393,434,449,463) and
 * torch_scatter `scatter_mean(messages, row, ...)` (Models/BuckGNN.py:561).
 *
 * Stable counting sort of the E edges by key row (key_row = 1: by target
 * edge_index[1], the SAGEConv direction; key_row = 0: by edge_index[0], the
 * GraphNetBlock direction):
 *    perm   == argsort(key, stable)            [E]   int32
 *    rowptr == concat(0, cumsum(bincount(key, N)))  [N+1] int32
 *    col[i] == other_row[perm[i]]              [E]   int32
 * bit-exact.  Rows whose degree exceeds BG_BIG_ROW_THRESHOLD (the super-node hub
 * rows) are additionally listed in big_rows (unordered), their count in info[1].
 *    info[0] : bit 0 set if any index was outside [0, N)   (such edges are dropped)
 *    info[1] : number of big rows
 *    info[4] : number of big rows that are NOT "range hubs" (see below) or whose ranges overlap
 *    info[5] : largest big-row degree
 *    info[6] : 1 if any row has no entries (a node without in-edges), else 0
 * (info has 8 words; bg_batch_info conventionally writes words 2-3 of the same buffer.)
 * big_rows must hold bg_csr_max_big_rows(E) entries.  E, N < 2^31.
 * hub_lo [bg_csr_max_big_rows(E)] and hub_of_row [N] (optional, both or neither): a big row whose
 * sorted neighbour list is exactly lo, lo+1, ..., lo+deg-1 (the reference's super node) gets
 * hub_lo[b] = lo and hub_of_row[j] = b for every j in that range, else hub_lo[b] = -1; rows in no
 * range keep hub_of_row = -1.  bg_sage_aggregate uses this to fold hub rows into its row pass.
 */
#define BG_BIG_ROW_THRESHOLD 64
int64_t bg_csr_max_big_rows(int64_t n_edges);
int bg_csr_workspace_bytes(int64_t n_nodes, int64_t n_edges, size_t* bytes_host);
int bg_csr_build(const int64_t* edge_index, int64_t n_edges, int64_t n_nodes, int key_row,
                 int32_t* rowptr, int32_t* col, int32_t* perm, int32_t* big_rows, int32_t* info,
                 int32_t* hub_lo, int32_t* hub_of_row,
                 void* workspace, size_t workspace_bytes, void* stream);

/* Graph offsets from the PyG `batch` vector; replaces the index handling inside
 * `global_mean_pool(x, batch)` (Models/BuckGNN.py:274).
 * bg_batch_info:  info[0] = batch[N-1] + 1 (= batch.max()+1 for sorted batch),
 *                 info[1] = 1 if batch is not non-decreasing or has a negative id.
 * bg_graph_ptr_build: graph_ptr[g] = first node index with batch >= g, g in [0, G];
 *                 graph_ptr[G] = N.  Requires sorted batch (PyG DataLoader order). */
int bg_batch_info(const int64_t* batch, int64_t n_nodes, int32_t* info, void* stream);
/* Copies n <= 256 device words to PINNED host memory (UVA-mapped, e.g. torch pin_memory) with SM stores +
 * a system fence: the host reads them after an event recorded behind this call.  Unlike a D2H memcpy it
 * cannot queue on a copy engine behind the H2D transfer of the next batch (the forward's only host sync,
 * PyG's `batch.max()+1` equivalent, stays off the PCIe copy queues). */
int bg_publish_words(const int32_t* src, int32_t* dst_host_mapped, int32_t n, void* stream);
int bg_graph_ptr_build(const int64_t* batch, int64_t n_nodes, int64_t n_graphs, int32_t* graph_ptr,
                       void* stream);

/* ------------------------------------------------------------------ K5: node encoder front
 * First two Linear+ReLU of `node_encoder` (Models/BuckGNN.py:68-72, applied :323):
 *    h = relu(relu(x W1^T + b1) W2^T + b2),  x [N,F] f32 -> h [N,128] (out_dtype)
 * W1 [64,F], W2 [128,64] f32 row-major (out,in) as in nn.Linear.  F <= 32.
 * row_gather (optional, DEVICE [N] int32): output row i is computed from input row row_gather[i]
 * (the edge encoder reads `edge_attr` through the CSR permutation this way).
 * nonfinite_flag (optional, DEVICE int32): OR-ed with 1 when a 16-bit output cannot hold a value of h (fp16: above
 * 65504, or NaN) -- h is the one activation stored before any normalisation; pass the same word to bg_pool_head. */
int bg_encoder_front(const float* x, int64_t n_nodes, int32_t n_features,
                     const float* w1, const float* b1, const float* w2, const float* b2,
                     const int32_t* row_gather, void* out, int out_dtype, int32_t* nonfinite_flag, void* stream);

/* ------------------------------------------------------------------ K2: neighbourhood aggregation
 * Replaces `x[src]` gather + `scatter_add_` + divide inside SAGEConv.propagate:
 *    out[i] = reduce_{e: key(e)=i} x[col(e)]     mean: sum / max(deg,1); max: 0 if deg = 0
 * x, out: [N,width] of `dtype` (bf16, f16 or f32), width 512 or 128 (the encoder's hidden layer, for the
 * folded first layer); accumulation in fp32 in CSR (stable) order.
 * Big rows (info[1] of bg_csr_build, read back by the host) are split across CTAs;
 * workspace from bg_aggregate_workspace_bytes(n_big).
 * hub_lo / hub_of_row (optional, both or neither; from bg_csr_build, valid only when its info[4] == 0)
 * with hub_max_degree = info[5]: every big row is a "range hub", and for width 512 and mean / sum
 * aggregation the hub rows are folded into the row pass (each row is added to its hub's partial sum
 * while it is in cache) instead of a second pass over x.  Workspace then from
 * bg_hubfold_workspace_bytes.  Summation order of a hub row is then (band, warp, row) instead of
 * CSR order; both are fixed, so results stay run-to-run deterministic. */
int bg_aggregate_workspace_bytes(int32_t n_big, size_t* bytes_host);
int bg_hubfold_workspace_bytes(int64_t n_nodes, int dtype, int32_t n_big, int32_t hub_max_degree,
                               size_t* bytes_host);
int bg_sage_aggregate(const void* x, void* out, int dtype, int64_t n_nodes, int32_t width,
                      const int32_t* rowptr, const int32_t* col,
                      const int32_t* big_rows, int32_t n_big, int aggr,
                      const int32_t* hub_lo, const int32_t* hub_of_row, int32_t hub_max_degree,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ K3: tensor-core update GEMM
 * out[m, 0:512] = epilogue( sum_s A_s[m, :] . B_s[:, :]^T )
 * Each segment s contributes A_s [M, k_s] times B_s [512, k_s] (nn.Linear weight
 * layout, K-major) -- the SAGE update is the two segments (agg, lin_l.weight),
 * (x, lin_r.weight), i.e. the concatenated [lin_l | lin_r] GEMM with K = 1024.
 * Replaces `lin_l(agg) + lin_r(x)`, `F.normalize`, `BatchNorm1d` (eval), `ReLU`
 * and the skip connection (Models/BuckGNN.py:449-457 and PyG SAGEConv.forward).
 * Epilogue order (each step optional):
 *    v = acc + bias;   v += G0[gidx0[m], :] + G1[gidx1[m], :];
 *    v /= max(||v||_2, 1e-12);  v = v*bn_scale + bn_shift;  v = max(v, 0);  v += residual[m, :]
 * The gathered addends serve the EA-GNN block (Models/BuckGNN.py:556-560), where
 * cat[x[row], x[col], e] W^T is evaluated as (x W_a^T)[row] + (x W_b^T)[col] + e W_c^T: the two
 * node-level products are gathered per edge inside the epilogue of the edge-level GEMM.
 * normalize cannot be combined with gathered addends, nor gathered addends with residual; gather[1] needs gather[0].
 * Rounding of the gathered addends with a 16-bit out_dtype (unlike bg_gemm128_gathered, which rounds once):
 * acc + bias is rounded to out_dtype first; two gathered rows are summed in out_dtype (one rounding) before they
 * join; without BatchNorm vectors the join is itself an out_dtype add (rounded again), with them it is an fp32 add
 * and the result is rounded once more at the store.  An fp32 out_dtype adds everything in fp32.
 * Operand formats: a_dtype == b_dtype in {BG_BF16, BG_F16} (tcgen05 kind::f16, k_s % 64 == 0;
 * the hardware rejects bf16 x fp16 mixes) or both BG_F32 (read as
 * tf32, kind::tf32; k_s % 32 == 0 -- with hi/lo split operands from bg_split_tf32 this
 * is the 3xTF32 "fp32-GEMM" mode).  fp32 accumulation in TMEM always.
 * out/residual dtype = out_dtype (any bg_dtype).  All base pointers 16-byte aligned, ld* such that
 * rows are 16-byte aligned.  cta_group must be 2 (tcgen05 cta_group::2 CTA pairs). */
#define BG_MAX_GEMM_SEGMENTS 8
typedef struct bg_gemm_segment {
  const void* a; int64_t lda;
  const void* b; int64_t ldb;
  int32_t k;
  int32_t b_groups;            /* 0 / 1: B is [512, k].  g > 1 (split-K weight gradients): B is [g*512, k], A is   */
                               /* [g*512, k] (m == g*512) and rows [i*512, +512) of A multiply rows [i*512, +512)  */
                               /* of B -- g independent 512 x 512 products in one launch; same g in every segment. */
} bg_gemm_segment;

typedef struct bg_epilogue {
  const float* bias_host;      /* [512] HOST pointers: the vectors travel in the kernel   */
  const float* bn_scale_host;  /* parameters (constant bank); NULL = absent                */
  const float* bn_shift_host;  /* required iff bn_scale_host is given                      */
  const void* residual;        /* DEVICE [M,512], ld = ldr, dtype = out_dtype, or NULL     */
  int64_t ldr;
  int32_t normalize;           /* F.normalize(p=2, dim=-1, eps=1e-12) */
  int32_t relu;
  const void* gather[2];       /* DEVICE [*,512] matrices of out_dtype (ld = gather_ld), NULL = absent */
  const int32_t* gather_idx[2];/* DEVICE [M] row index into gather[k]                      */
  int64_t gather_ld;
  float* inv_norm_out;         /* DEVICE [M] f32 or NULL: with normalize, 1 / max(||v||_2, 1e-12) per row (the   */
                               /* training forward saves it for the backward of F.normalize)                     */
  float* pool_block_sums;      /* DEVICE [ceil(M/32), 512] f32 or NULL.  Pool-fused epilogue for the LAST layer  */
                               /* of a graph-level model, whose output only feeds global_mean_pool               */
                               /* (Models/BuckGNN.py:515): the column sums of every 32-row block of the output   */
                               /* rows (the rounded values a store would have written; fp32, fixed order) are    */
                               /* written here, and only the blocks flagged in pool_block_keep are stored to     */
                               /* `out`.  Needs normalize, a 16-bit out_dtype, no residual / gathered addends.   */
  const uint8_t* pool_block_keep; /* DEVICE [ceil(M/32)] from bg_pool_block_flags; required with pool_block_sums */
} bg_epilogue;

int bg_gemm512(const bg_gemm_segment* segments_host, int32_t n_segments, int64_t m,
               int a_dtype, int b_dtype, const bg_epilogue* epilogue_host,
               void* out, int out_dtype, int64_t ldo, int cta_group, void* stream);

/* The fused SAGE layer (reference: SAGEConv.propagate + lin_l / lin_r + F.normalize + BatchNorm1d + ReLU + skip,
 * Models/BuckGNN.py:449-457, in ONE kernel): bg_gemm512 whose segment 0 is (aggregate_of(x), lin_l.weight) with K = 512
 * -- segment 0's `a` is ignored: four gather warps per CTA build the aggregate rows of the CTA's 128 nodes straight into
 * the shared-memory operand tile the tensor core reads (fp32 accumulation in CSR order, the same rounding as
 * bg_sage_aggregate: the operand is bit-identical), so the [N,512] aggregate matrix never exists in global memory.
 * Segment 1.. as in bg_gemm512 (the root rows: (x, lin_r.weight)).  16-bit activations; the epilogue must normalize
 * (skip rows and the pool-fused variant allowed, no gathered addends).  Rows whose degree exceeds
 * BG_BIG_ROW_THRESHOLD take their aggregate from hub_agg (bg_sage_aggregate_hubs). */
typedef struct bg_fused_aggregate {
  const void* x; int64_t ldx;     /* DEVICE [N,512] rows of a_dtype: the layer input */
  const int32_t* rowptr;          /* CSR by target (bg_csr_build, key_row = 1) */
  const int32_t* col;
  int32_t aggr;                   /* BG_AGGR_MEAN or BG_AGGR_SUM */
  int32_t n_big;
  const void* hub_agg;            /* DEVICE [n_big, 512] of a_dtype, row b = aggregate of node big_rows[b]; NULL iff n_big == 0 */
  const int32_t* big_rows;
} bg_fused_aggregate;

int bg_sage_fused512(const bg_gemm_segment* segments_host, int32_t n_segments, int64_t m,
                     int a_dtype, int b_dtype, const bg_epilogue* epilogue_host, const bg_fused_aggregate* fused_host,
                     void* out, int out_dtype, int64_t ldo, void* stream);

/* The update GEMM at width 128 (a model with hidden_channels = 128, the reference's default):
 *    out[m, 0:128] = epilogue( sum_s A_s[m, :] . B_s[:, :]^T ),   B_s [128, k_s] (nn.Linear weight layout)
 * Same arguments, operand formats, K rules and epilogue order as bg_gemm512, with 128 for 512 throughout: the
 * epilogue's host vectors are [128], residual / out rows are [M,128] (ld >= 128), pool_block_sums is [ceil(M/32), 128].
 * Not built at this width (BG_ERR_UNSUPPORTED): gathered addends (see bg_gemm128_gathered) and b_groups > 1. */
int bg_gemm128(const bg_gemm_segment* segments_host, int32_t n_segments, int64_t m,
               int a_dtype, int b_dtype, const bg_epilogue* epilogue_host,
               void* out, int out_dtype, int64_t ldo, int cta_group, void* stream);

/* bg_gemm128 with gathered pre-activation addends (the edge GEMMs of a hidden_channels = 128 EA-GNN layer, GraphNetBlock
 * Models/BuckGNN.py:528-566):
 *    out[m, :] = relu( sum_s A_s[m, :] . B_s^T + bias + gather[0][gather_idx[0][m], :] + gather[1][gather_idx[1][m], :] )
 * summed in fp32 and rounded once to out_dtype.  gather[k] are DEVICE [*, 128] row-major matrices of out_dtype with
 * leading dimension gather_ld >= 128 (rows 16-byte aligned), gather_idx[k] DEVICE [M] int32 row indices; gather[1] may
 * be NULL.  BG_ERR_INVALID for a missing index, gather[1] without gather[0] or a misaligned matrix;
 * BG_ERR_UNSUPPORTED for gathered addends together with normalize, residual or the pool-fused epilogue (as bg_gemm512).
 * Without gathered addends the call is bg_gemm128.  Every argument is checked before the first CUDA call. */
int bg_gemm128_gathered(const bg_gemm_segment* segments_host, int32_t n_segments, int64_t m,
                        int a_dtype, int b_dtype, const bg_epilogue* epilogue_host,
                        void* out, int out_dtype, int64_t ldo, int cta_group, void* stream);

/* Aggregates of the hub rows only, compact: hub_out[b, :] = reduce over the neighbours of node big_rows[b] (mean / sum,
 * 16-bit rows).  workspace: bg_aggregate_workspace_bytes(n_big). */
int bg_sage_aggregate_hubs(const void* x, int dtype, const int32_t* rowptr, const int32_t* col, const int32_t* big_rows,
                           int32_t n_big, int aggr, void* hub_out, void* workspace, size_t workspace_bytes, void* stream);

/* Weight gradients of a Linear with 512 outputs, dW[o, i] = sum_n dz[n, o] * act[n, i] (autograd of lin_l / lin_r,
 * Models/BuckGNN.py:449): the reduction runs over the ROWS of the row-major dz [n_rows, 512] and act [n_rows, act_cols]
 * (act_cols <= 512; dW columns beyond it come out 0), i.e. both tcgen05 operands are MN-major -- TMA reads them where
 * they lie, no transposed copies (f32 = tf32 operands use the 32-byte-atom swizzle).
 * Split over the nodes: chunk s covers rows [s*chunk_k, (s+1)*chunk_k) (chunk_k a multiple of 64, n_chunks*chunk_k
 * >= n_rows, rows beyond n_rows read as zero) and writes partial[s] ([512, 512] f32); sum the chunks with
 * bg_reduce_partials.  One 256 x 512 output tile per CTA pair: n_chunks = 37 fills a B200. */
int bg_wgrad512(const void* dz, int64_t ld_dz, const void* act, int32_t act_cols, int64_t ld_act, int dtype,
                int64_t n_rows, int32_t n_chunks, int64_t chunk_k, float* partial, void* stream);

/* ------------------------------------------------------------------ K4: pooling + regression head
 * Replaces `get_pooling_layer` + `decoder(pooled).squeeze()` (Models/BuckGNN.py:246-307, 515-516):
 *    BG_POOL_MEAN                   pooled[g] = sum_{i in g} x[i] / max(count_g, 1)          (:274)
 *    BG_POOL_MEAN_NO_SUPER          same over all nodes but the graph's last (super) node    (:277-282)
 *    BG_POOL_SUPERNODE_ONLY         pooled[g] = x[last node of g]                            (:283-284)
 *    BG_POOL_SUPERNODE_WITH_POOLING cat[mean_no_super, super]  (1024 wide)                   (:285-293)
 * pre_w/pre_b [512,512]/[512] non-NULL: the `MLPPooling` Linear+ReLU on the mean (:294-305, 568-581);
 * allowed with the two mean modes only.  Then decoder Linear(in,128) ReLU Linear(128,64) ReLU
 * Linear(64,out_dim), in = 1024 for SUPERNODE_WITH_POOLING else 512; all weights f32, nn.Linear layout.
 * x [N,512] of `dtype`; pred [G,out_dim] f32; pooled_out [G,in] f32 optional (NULL to skip).
 * workspace from bg_pool_workspace_bytes(G).
 * nonfinite_flag (optional, DEVICE int32): when the word is non-zero at kernel time every prediction is written as
 * NaN (an upstream kernel overflowed its 16-bit storage: fail loudly, without a host sync). */
typedef enum bg_pool_mode {
  BG_POOL_MEAN = 0, BG_POOL_MEAN_NO_SUPER = 1, BG_POOL_SUPERNODE_ONLY = 2, BG_POOL_SUPERNODE_WITH_POOLING = 3
} bg_pool_mode;
int bg_pool_workspace_bytes(int64_t n_graphs, size_t* bytes_host);
int bg_pool_head(const void* x, int dtype, int64_t n_nodes, const int32_t* graph_ptr, int64_t n_graphs,
                 int pool_mode, const float* pre_w, const float* pre_b,
                 const float* w1, const float* b1, const float* w2, const float* b2,
                 const float* w3, const float* b3, int32_t out_dim,
                 float* pred, float* pooled_out,
                 void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream);

/* Pooling over the block sums of a pool-fused bg_gemm512 (bg_epilogue.pool_block_sums): same result and arguments
 * as bg_pool_head, but x holds valid rows only in the blocks flagged by bg_pool_block_flags -- keep[b] = 1 for every
 * 32-row block [32b, 32b+32) that contains the first or the last row of a graph (so every other block lies inside one
 * graph, and the super node's row -- the graph's last -- is always stored).  16-bit x only.  The row sums are added in
 * a different (fixed) order than bg_pool_head's, so predictions agree to fp32 rounding, not bit for bit. */
int bg_pool_block_flags(const int32_t* graph_ptr, int64_t n_graphs, int64_t n_nodes, uint8_t* keep, void* stream);
int bg_pool_head_blocks(const void* x, int dtype, int64_t n_nodes, const int32_t* graph_ptr, int64_t n_graphs,
                        int pool_mode, const float* pre_w, const float* pre_b,
                        const float* w1, const float* b1, const float* w2, const float* b2,
                        const float* w3, const float* b3, int32_t out_dim,
                        float* pred, float* pooled_out, const float* block_sums, const uint8_t* keep,
                        void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream);

/* bg_pool_head / bg_pool_head_blocks for x [N,128] (hidden_channels = 128): same arguments and pooling modes;
 * the pooled feature is 128 wide (256 for BG_POOL_SUPERNODE_WITH_POOLING), pre_w / pre_b are [128,128] / [128],
 * w1 is [128, in], block_sums [ceil(N/32), 128].  The decoder is the same 3-layer head: a 2-layer
 * Linear(in,64) ReLU Linear(64,out) runs exactly as w1 = [W1; 0] (rows padded to 128), b1 = [b1; 0], w2 = [I64 | 0],
 * b2 = 0, w3 = W2, b3 = b2. */
int bg_pool_head128(const void* x, int dtype, int64_t n_nodes, const int32_t* graph_ptr, int64_t n_graphs,
                    int pool_mode, const float* pre_w, const float* pre_b,
                    const float* w1, const float* b1, const float* w2, const float* b2,
                    const float* w3, const float* b3, int32_t out_dim,
                    float* pred, float* pooled_out,
                    void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream);
int bg_pool_head_blocks128(const void* x, int dtype, int64_t n_nodes, const int32_t* graph_ptr, int64_t n_graphs,
                           int pool_mode, const float* pre_w, const float* pre_b,
                           const float* w1, const float* b1, const float* w2, const float* b2,
                           const float* w3, const float* b3, int32_t out_dim,
                           float* pred, float* pooled_out, const float* block_sums, const uint8_t* keep,
                           void* workspace, size_t workspace_bytes, const int32_t* nonfinite_flag, void* stream);

/* Node-level decoder of a hidden_channels = 128 model (Models/BuckGNN.py:518-524, h <= 128 decoder :41-65):
 *   out[r] = W2 relu(W1 x[r] + b1) + b2      x [n_rows,128] of `dtype`, out [n_rows,out_dim] f32 row-major
 * w1 [64,128] in the operand format of dtype (fp16 / bf16 for 16-bit x, f32 for f32 x), b1 [64] f32,
 * w2 [out_dim,64] f32, b2 [out_dim] f32, 1 <= out_dim <= 8.  Rows are independent; no workspace, no atomics.
 * 16-bit x: mma.sync with fp32 accumulation, the hidden layer kept in fp32 (not rounded); f32 x: fp32 FMAs.
 * x and w1 16-byte aligned, b1 / w2 / b2 / out 4-byte aligned.  n_rows == 0 launches nothing (x and out may then be
 * NULL).  The result is the same bit for bit from run to run. */
int bg_node_head128(const void* x, int dtype, int64_t n_rows, const void* w1, const float* b1,
                    const float* w2, const float* b2, int32_t out_dim, float* out, void* stream);

/* ------------------------------------------------------------------ EA-GNN helpers
 * bg_expand_rowptr: row_of[i] = r with rowptr[r] <= i < rowptr[r+1], iota[i] = i   (i < E)
 *   (row ids of the CSR slots, and the identity "col" that turns bg_sage_aggregate into the
 *   segmented mean torch_scatter.scatter_mean(messages, row) needs once edges are in CSR order);
 *   row_of / iota may be NULL.
 *   nonempty (optional, [n_rows, 64] of nonempty_dtype): column 0 = 1 for rows with >= 1 entry, rest 0;
 *   with as_count != 0 columns 0..2 hold the row's entry count as base-256 digits (count = c0 + 256 c1 + 65536 c2:
 *   each digit is exact in bf16 / fp16 / tf32, a super node's degree is not) --
 *   a K = 64 GEMM segment that applies a bias only to rows whose scatter_mean segment is non-empty
 *   (what remains of phi's second-layer bias after that Linear is folded through the mean).
 * bg_add: out = a + b (+ c) elementwise over n values of `dtype`, fp32 math (skip connections
 *   of the EA-GNN wrapper, Models/BuckGNN.py:382-384). */
int bg_expand_rowptr(const int32_t* rowptr, int64_t n_rows, int64_t n_entries, int32_t* row_of, int32_t* iota,
                     void* nonempty, int nonempty_dtype, int as_count, void* stream);
int bg_add(const void* a, const void* b, const void* c_or_null, void* out, int dtype, int64_t n, void* stream);

/* ------------------------------------------------------------------ SAGPooling (SURVEY.md section 8 row f4)
 * Replaces PyG `SAGPooling(hidden, ratio=0.5, GNN=SAGEConv, aggr='add')` of the `GraphSAGE_SAG` / `EAGNN_SAG`
 * variants (constructed Models/BuckGNN.py:203-208, 231-236; applied :365-367, :502-504):
 *    s      = tanh(sign * (w_l . sum_{j -> i} x_j + bias + w_r . x_i))      score GNN = SAGEConv(512, 1, aggr='add')
 *    perm   = for each graph its ceil(ratio * n_g) highest-scoring nodes, descending score, ties by lower node id
 *    x'     = x[perm] * s[perm];  batch' = batch[perm];  edge_index' = edges whose two endpoints are kept,
 *             relabelled to the new row ids, original order (PyG `topk` / `filter_adj`).
 * bg_sag_select (x [N,512] of `dtype`; rowptr/col/big_rows/n_big: bg_csr_build keyed by TARGET, key_row = 1;
 *   w_l, w_r [512] f32 device = pool.gnn.lin_l.weight / lin_r.weight, bias = pool.gnn.lin_l.bias; sign = +1, or
 *   the sign of `pool.select.weight` for checkpoints of PyG >= 2.4 whose SelectTopK rescales the score):
 *    score [N] f32;  new_id [N] int32 = new row of a kept node, -1 for a dropped one;  perm [N'] int32 (buffer of N);
 *    batch_out [N'] int64;  score_out [N'] f32 = s[perm];  new_graph_ptr [G+1] int32;
 *    info[0] = N' (kept nodes), info[1] = E' (kept edges) -- read them back (bg_publish_words) before bg_sag_connect.
 * bg_sag_connect: edge_index_out [2, E'] int64, kept_edge [E'] int32 (nullable) = original edge id of each kept
 *   edge.  `workspace` must be the buffer bg_sag_select used, untouched in between (it holds the block offsets).
 * bg_gather_rows: out[r, 0:512] = x[row_index[r], 0:512] * (row_scale ? row_scale[row_index[r]] : 1)  --
 *   x[perm] * score[perm], and the edge-feature rows of the kept edges for EAGNN_SAG.  A negative row_index[r] gives
 *   a zero row (the training step scatters edge gradients back this way: dropped edges receive none).
 * bg_index_invert: out[perm[i]] = i;  bg_index_gather: out[i] = table[idx[i]]   (int32 index plumbing). */
int bg_sag_workspace_bytes(int64_t n_nodes, int64_t n_edges, int64_t n_graphs, size_t* bytes_host);
int bg_sag_select(const void* x, int dtype, int64_t n_nodes, const int32_t* rowptr, const int32_t* col,
                  const int32_t* big_rows, int32_t n_big, const float* w_l, const float* w_r, float bias, float sign,
                  const int32_t* graph_ptr, int64_t n_graphs, float ratio, const int64_t* edge_index, int64_t n_edges,
                  float* score, int32_t* new_id, int32_t* perm, int64_t* batch_out, float* score_out,
                  int32_t* new_graph_ptr, int32_t* info, void* workspace, size_t workspace_bytes, void* stream);
int bg_sag_connect(const int64_t* edge_index, int64_t n_edges, int64_t n_nodes, const int32_t* new_id,
                   int64_t n_edges_out, int64_t* edge_index_out, int32_t* kept_edge,
                   void* workspace, size_t workspace_bytes, void* stream);
/* Backward of SAGPooling for the training step (autograd of `self.pool`, Models/BuckGNN.py:502-504): given
 * dx_pooled = d loss / d x' [N', 512], x [N, 512] (the pooling input), perm / new_id / score [N] (= all scores) from
 * bg_sag_select and the CSR of the un-pooled graph keyed by SOURCE (bg_csr_build key_row = 0, with its big rows):
 *    dpre_j = sign (1 - s_j^2) (dx'_r . x_j) for j = perm[r], 0 for dropped nodes      (tanh and the row scaling)
 *    t_j    = sum_{i: j -> i} dpre_i                                                   (the 'add' aggregation, transposed)
 *    dx_j   = [j kept] s_j dx'_{new_id[j]} + w_l t_j + w_r dpre_j                      [N, 512] of `dtype`
 * t, dpre [N] f32 are outputs too: the scorer's gradients are dw_l = sum_j t_j x_j, dw_r = sum_j dpre_j x_j
 * (bg_sgemm with m = 1) and db = sum_j dpre_j (bg_colsum). */
int bg_sag_pool_backward(const void* dx_pooled, const void* x, int dtype, int64_t n_nodes, int64_t n_nodes_out,
                         const int32_t* perm, const int32_t* new_id, const float* score, float sign,
                         const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_rows_src,
                         int32_t n_big_src, const float* w_l, const float* w_r, void* dx, float* t, float* dpre,
                         void* stream);
int bg_gather_rows(const void* x, int dtype, int64_t ldx, const int32_t* row_index, const float* row_scale,
                   int64_t n_rows_out, void* out, int64_t ldo, void* stream);
int bg_index_invert(const int32_t* perm, int64_t n, int32_t* out, void* stream);
int bg_index_gather(const int32_t* table, const int32_t* idx, int64_t n, int32_t* out, void* stream);
/* SAGPooling of a hidden_channels = 128 model (BuckGNN.native128_sag), on [*, 128] rows: every argument and rule is the
 * one of the 512-wide call above, with 128 for 512 --
 *   bg_sag_select128: x [N,128], w_l / w_r [128].  Only the pass computing w_l . x and w_r . x reads rows; the score,
 *     the top-k, the new offsets and the edge count are the 512-wide call's, and bg_sag_connect /
 *     bg_sag_workspace_bytes serve both widths.
 *   bg_gather_rows128: out[r, 0:128] = x[row_index[r], 0:128] * (row_scale ? row_scale[row_index[r]] : 1), ldx / ldo
 *     >= 128; a negative row_index[r] gives a zero row.
 *   bg_sag_pool_backward128: dx_pooled [N',128], x / dx [N,128], w_l / w_r [128]; t and dpre stay [N].
 * Every argument is checked before the first CUDA call.  fp32 accumulation in a fixed order, no floating-point atomics:
 * repeated calls are bit-identical. */
int bg_sag_select128(const void* x, int dtype, int64_t n_nodes, const int32_t* rowptr, const int32_t* col,
                     const int32_t* big_rows, int32_t n_big, const float* w_l, const float* w_r, float bias, float sign,
                     const int32_t* graph_ptr, int64_t n_graphs, float ratio, const int64_t* edge_index, int64_t n_edges,
                     float* score, int32_t* new_id, int32_t* perm, int64_t* batch_out, float* score_out,
                     int32_t* new_graph_ptr, int32_t* info, void* workspace, size_t workspace_bytes, void* stream);
int bg_gather_rows128(const void* x, int dtype, int64_t ldx, const int32_t* row_index, const float* row_scale,
                      int64_t n_rows_out, void* out, int64_t ldo, void* stream);
int bg_sag_pool_backward128(const void* dx_pooled, const void* x, int dtype, int64_t n_nodes, int64_t n_nodes_out,
                            const int32_t* perm, const int32_t* new_id, const float* score, float sign,
                            const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_rows_src,
                            int32_t n_big_src, const float* w_l, const float* w_r, void* dx, float* t, float* dpre,
                            void* stream);

/* ------------------------------------------------------------------ training step
 * What `loss.backward()` and train-mode BatchNorm1d / Dropout need around the forward kernels
 * (TRAIN_FINAL.py:289-297 driving Models/BuckGNN.py:445-458 with model.train()).  Per GraphSAGE layer:
 *   forward:  agg = bg_sage_aggregate(x);  u = bg_gemm512(normalize, inv_norm_out) -- no BN in the epilogue;
 *             bg_bn_batch_stats(u) -> a, shift (+ running statistics);  y = bg_bn_act_forward(u, x_prev)
 *   backward: bg_sage_backward_rows(u, dy) -> dz (+ dgamma, dbeta);  dagg = bg_gemm512(dz_scaled, Wl^T rows);
 *             s = bg_sage_aggregate over the CSR keyed by SOURCE (A^T);  dx = bg_gemm512(dz, Wr^T rows) + s;
 *             dWl = dz^T agg, dWr = dz^T x: bg_transpose_chunks + bg_gemm512(b_groups) + bg_reduce_partials.
 * Every reduction is two-stage in a fixed order (no floating-point atomics).
 *
 * bg_bn_batch_stats: batch mean / biased variance of the N rows of u [N,512] (torch BatchNorm1d, train mode):
 *   a = gamma / sqrt(var + eps), shift = beta - mean * a, mean, invstd = 1/sqrt(var + eps)   (f32 [512], device);
 *   running_mean / running_var (nullable) updated with `momentum` (unbiased variance), *num_batches_tracked += 1.
 * bg_bn_act_forward: y = dropout(relu(a * u + shift) + x_prev)   (Models/BuckGNN.py:451-458; x_prev nullable).
 *   Dropout is counter-based: element (r, c) is kept iff hash(seed, r*512 + c) >= dropout_p * 2^32, kept values
 *   are scaled by 1/(1-p); the backward pass regenerates the mask from the same seed.  Without BatchNorm
 *   (GraphSage_addAggr_Shared) pass a = 1, shift = 0.
 * bg_sage_backward_rows: g = dropout'(dy + dy2);  dv = g * [a*u + shift > 0];
 *   dbeta (+)= sum_r dv;  dgamma (+)= sum_r dv * (u - mean) * invstd          (mean == NULL: no BatchNorm)
 *   du = BatchNorm1d input gradient;  dz = inv_norm * (du - u * (u . du))       (F.normalize backward)
 *   dz_scaled (nullable) = dz / max(deg, 1) with deg from rowptr (mean aggregation);  g_out (nullable) = g.
 *   workspace from bg_train_workspace_bytes(N). */
int bg_train_workspace_bytes(int64_t n_rows, size_t* bytes_host);
int bg_bn_batch_stats(const void* u, int dtype, int64_t n_rows, const float* gamma, const float* beta, float eps,
                      float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                      float* a_out, float* shift_out, float* mean_out, float* invstd_out,
                      void* workspace, size_t workspace_bytes, void* stream);
int bg_bn_act_forward(const void* u, const void* x_prev, void* y, int dtype, int64_t n_rows, const float* a,
                      const float* shift, float dropout_p, uint64_t seed, void* stream);
int bg_sage_backward_rows(const void* u, const void* dy, const void* dy2, const float* inv_norm, const int32_t* rowptr,
                          int dtype, int64_t n_rows, const float* a, const float* shift, const float* mean,
                          const float* invstd, float dropout_p, uint64_t seed, float* dgamma, float* dbeta,
                          int accumulate, void* dz, void* dz_scaled, void* g_out,
                          void* workspace, size_t workspace_bytes, void* stream);
/* Split-K operand layout for the weight gradients: out[s][c][j] = in[s*chunk_k + j][c] (0 beyond n_rows), i.e.
 * n_chunks K-major [n_cols, chunk_k] matrices; n_cols and chunk_k multiples of 32, n_chunks*chunk_k >= n_rows.
 * out_rows_per_chunk (0 = n_cols) > n_cols places chunk s at row s*out_rows_per_chunk of out (a narrow matrix
 * padded to 512 rows per chunk; the caller zero-fills out first).
 * bg_reduce_partials: out[i] (+)= sum_s partial[s][i]. */
int bg_transpose_chunks(const void* in, int dtype, int64_t n_rows, int32_t n_cols, int64_t ld, int32_t n_chunks,
                        int64_t chunk_k, int32_t out_rows_per_chunk, void* out, void* stream);
/* out[m, n] (f32, contiguous [M, n_cols]) = in[m, n] * [mask[m, n] > 0] (mask nullable): ReLU backward while
 * narrowing the [M, 512] output of a zero-padded bg_gemm512 to its n_cols real columns (encoder gradients). */
int bg_mask_narrow(const void* in, int in_dtype, int64_t ld_in, const void* mask, int mask_dtype, int64_t ld_mask,
                   int64_t m, int32_t n_cols, float* out, void* stream);
int bg_reduce_partials(const float* partial, int32_t n_chunks, int64_t n, float* out, int accumulate, void* stream);
/* out[c] (+)= sum_r in[r, c]  (bias gradients). */
int bg_colsum_workspace_bytes(int64_t rows, int32_t cols, size_t* bytes_host);
int bg_colsum(const void* in, int dtype, int64_t rows, int32_t cols, int64_t ld, float* out, int accumulate,
              void* workspace, size_t workspace_bytes, void* stream);
/* get_pooling_layer backward (Models/BuckGNN.py:273-293): dx[r] = dpooled[graph(r)] * w(r) for every bg_pool_mode;
 * dpooled [G, >= 512] f32 (ld = ldp), [G, 1024] for BG_POOL_SUPERNODE_WITH_POOLING. */
int bg_pool_backward(const float* dpooled, int64_t ldp, const int32_t* graph_ptr, int64_t n_graphs, int pool_mode,
                     int64_t n_nodes, void* dx, int dtype, void* stream);
/* fp32 GEMM on the CUDA cores for the narrow layers (encoder 16->64->128, decoder 512->128->64->out and their
 * gradients; ~2 % of a step's flops):  out[m,n] (+)= mask( relu( sum_k A(m,k) B(k,n) + bias[n] ) ),
 * A(m,k) = a[m*sam + k*sak], B(k,n) = b[k*sbk + n*sbn] (any bg_dtype, element strides), mask (nullable):
 * out = 0 where mask[m,n] <= 0 (ReLU backward).  Split-K, reduced in a fixed order. */
int bg_sgemm_workspace_bytes(int64_t m, int64_t n, int64_t k, size_t* bytes_host);
int bg_sgemm(const void* a, int a_dtype, int64_t sam, int64_t sak, const void* b, int b_dtype, int64_t sbk, int64_t sbn,
             int64_t m, int64_t n, int64_t k, const float* bias, int relu, const void* mask, int mask_dtype,
             int64_t mask_ld, void* out, int out_dtype, int64_t ldo, int accumulate,
             void* workspace, size_t workspace_bytes, void* stream);
/* Elementwise pieces of the EA-GNN training step ([n_rows, 512] node or edge tensors of `dtype`):
 * bg_dropout_residual: y = dropout(x + x_prev)  -- the wrapper's skip + Dropout, Models/BuckGNN.py:382-386 (x_prev nullable).
 * bg_grad_mask:        out = dropout'(dy + dy2) * [act > 0]  (dy2, act nullable; dropout_p = 0: none) -- Dropout and
 *                      ReLU backward in one pass.
 * bg_segment_expand:   out[s] = src[r] (/ count_r when mean != 0) for every CSR slot s of row r -- the backward of
 *                      torch_scatter.scatter_mean(messages, row) (:561) and of the row-gather x[row]. */
int bg_dropout_residual(const void* x, const void* x_prev, void* y, int dtype, int64_t n_rows, float dropout_p,
                        uint64_t seed, void* stream);
int bg_grad_mask(const void* dy, const void* dy2, const void* act, void* out, int dtype, int64_t n_rows, float dropout_p,
                 uint64_t seed, void* stream);
int bg_segment_expand(const void* src, const int32_t* rowptr, int64_t n_rows, int mean, void* out, int dtype, void* stream);

/* Backward of the 'max' neighbourhood aggregation (autograd of SAGEConv(aggr='max'), Models/BuckGNN.py:171-176, 459-471):
 * forward agg_i[c] = max_{j -> i} x_j[c] (0 without in-edges).  The gradient is the one autograd gives the reference
 * when PyG reduces with torch's scatter_reduce_('amax', include_self=False) on a zero-initialised output: dagg_i[c] is
 * shared evenly by the neighbours attaining the maximum, the zero-initialised element counting as one more sharer
 * when the maximum is 0:   n_i[c] = [agg_i[c] == 0] + #{j -> i: x_j[c] == agg_i[c]},
 *                          dx_j[c] = sum_{i: j -> i} [x_j[c] == agg_i[c]] dagg_i[c] / n_i[c].
 * x, agg, dagg, w_scratch, dx: [N, 512] of `dtype`; CSR keyed by target (bg_csr_build key_row = 1) and by source
 * (key_row = 0), each with its big-row list (hub rows are split over 8 CTAs whose partial sums go through `workspace`,
 * sized by bg_max_bwd_workspace_bytes).  No atomics: two gather passes, fixed summation order. */
int bg_max_bwd_workspace_bytes(int32_t n_big_tgt, int32_t n_big_src, size_t* bytes_host);
int bg_max_aggregate_backward(const void* x, const void* agg, const void* dagg, int dtype, int64_t n_nodes,
                              const int32_t* rowptr_tgt, const int32_t* col_tgt, const int32_t* big_rows_tgt, int32_t n_big_tgt,
                              const int32_t* rowptr_src, const int32_t* col_src, const int32_t* big_rows_src, int32_t n_big_src,
                              void* w_scratch, void* dx, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ training step at width 128
 * The same layer step for a hidden_channels = 128 model on rows [N, 128] (BuckGNN.native128_train): every argument and
 * rule is the one of the 512-wide entry point above, with 128 for 512 --
 *   bg_bn_batch_stats128, bg_bn_act_forward128, bg_sage_backward_rows128: u / x_prev / y / dy / dy2 / dz / dz_scaled /
 *     g_out [N, 128]; the BatchNorm vectors [128]; workspace from bg_train_workspace_bytes(N) (as at 512).  The dropout
 *     element index stays r*512 + c, so the mask is the first 128 columns of the 512-wide one (bg_dropout_mask).
 *   bg_pool_backward128: dx [N, 128]; dpooled [G, >= 128] (ld = ldp), [G, 256] for BG_POOL_SUPERNODE_WITH_POOLING.
 *   bg_max_aggregate_backward128: x, agg, dagg, w_scratch, dx [N, 128]; workspace from bg_max_bwd_workspace_bytes.
 * bg_wgrad128: both weight gradients of a 128-wide SAGE layer in one tcgen05 launch,
 *     dwl[o, i] (+)= sum_n dz[n, o] agg[n, i],   dwr[o, i] (+)= sum_n dz[n, o] x[n, i]     (f32 [128, 128] each)
 *   dz, agg, x: contiguous [n_rows, 128] of `dtype`, read in place as MN-major operands (no transposed copies; f32 =
 *   tf32 operands with the 32-byte-atom swizzle).  Split over the nodes as bg_wgrad512: chunk s covers rows
 *   [s*chunk_k, (s+1)*chunk_k), chunk_k a multiple of 64 (16-bit) / 32 (tf32), n_chunks*chunk_k >= n_rows; one
 *   256 x 128 tile [dWl^T ; dWr^T] per chunk and CTA pair goes to partial ([n_chunks * 256, 128] f32, caller-owned),
 *   then a second kernel sums the chunks in order and transposes.  accumulate != 0 adds into dwl / dwr.  No
 *   floating-point atomics: repeated calls are bit-identical. */
int bg_bn_batch_stats128(const void* u, int dtype, int64_t n_rows, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                         float* a_out, float* shift_out, float* mean_out, float* invstd_out,
                         void* workspace, size_t workspace_bytes, void* stream);
int bg_bn_act_forward128(const void* u, const void* x_prev, void* y, int dtype, int64_t n_rows, const float* a,
                         const float* shift, float dropout_p, uint64_t seed, void* stream);
int bg_sage_backward_rows128(const void* u, const void* dy, const void* dy2, const float* inv_norm, const int32_t* rowptr,
                             int dtype, int64_t n_rows, const float* a, const float* shift, const float* mean,
                             const float* invstd, float dropout_p, uint64_t seed, float* dgamma, float* dbeta,
                             int accumulate, void* dz, void* dz_scaled, void* g_out,
                             void* workspace, size_t workspace_bytes, void* stream);
int bg_pool_backward128(const float* dpooled, int64_t ldp, const int32_t* graph_ptr, int64_t n_graphs, int pool_mode,
                        int64_t n_nodes, void* dx, int dtype, void* stream);
int bg_max_aggregate_backward128(const void* x, const void* agg, const void* dagg, int dtype, int64_t n_nodes,
                                 const int32_t* rowptr_tgt, const int32_t* col_tgt, const int32_t* big_rows_tgt,
                                 int32_t n_big_tgt, const int32_t* rowptr_src, const int32_t* col_src,
                                 const int32_t* big_rows_src, int32_t n_big_src,
                                 void* w_scratch, void* dx, void* workspace, size_t workspace_bytes, void* stream);
int bg_wgrad128(const void* dz, const void* agg, const void* x, int dtype, int64_t n_rows, int32_t n_chunks,
                int64_t chunk_k, float* partial, float* dwl, float* dwr, int accumulate, void* stream);

/* The EA-GNN training step at width 128 (BuckGNN.native128_eagnn_train), on [N, 128] rows:
 *   bg_dropout_residual128, bg_grad_mask128, bg_segment_expand128: the arguments and rules of bg_dropout_residual,
 *     bg_grad_mask and bg_segment_expand with 128 for 512.  The dropout element index stays r*512 + c, so the mask is
 *     the first 128 columns of the 512-wide one (bg_dropout_mask).
 *   bg_wgrad128_ld: the weight gradients of EA-GNN's concatenated Linears, written in place into column slices,
 *       dw0[o * ld0 + i] (+)= sum_n dz[n, o] a0[n, i],   dw1[o * ld1 + i] (+)= sum_n dz[n, o] a1[n, i]    (o, i < 128)
 *     e.g. dw0 = dW + 128 with ld0 = 384 for the middle slice of a [128, 384] weight.  a1 is nullable (a single
 *     product; dw1 must then be null too), ld0 / ld1 >= 128.  dz, a0, a1, partial, n_chunks, chunk_k and accumulate as
 *     bg_wgrad128 (a single product still fills the 256 x 128 pair tile of partial: its second half is discarded). */
int bg_dropout_residual128(const void* x, const void* x_prev, void* y, int dtype, int64_t n_rows, float dropout_p,
                           uint64_t seed, void* stream);
int bg_grad_mask128(const void* dy, const void* dy2, const void* act, void* out, int dtype, int64_t n_rows, float dropout_p,
                    uint64_t seed, void* stream);
int bg_segment_expand128(const void* src, const int32_t* rowptr, int64_t n_rows, int mean, void* out, int dtype, void* stream);
int bg_wgrad128_ld(const void* dz, const void* a0, const void* a1, int dtype, int64_t n_rows, int32_t n_chunks,
                   int64_t chunk_k, float* partial, float* dw0, int64_t ld0, float* dw1, int64_t ld1, int accumulate,
                   void* stream);

/* Device-side collate (SURVEY.md section 8 row f1): PyG `DataLoader` / `Batch.from_data_list` for a dataset kept in HBM in
 * concatenated form -- x_all [sum n, F], ei_all [2, E_all] with node ids LOCAL to their graph (as
 * GraphCreate.py:417-432 emits them), ea_all [E_all, Fe], y_all [G_all], node_ptr / edge_ptr [G_all+1] int64.
 * bg_collate_ptr: out_node_ptr / out_edge_ptr [G+1] = exclusive scans of the sizes of the selected graphs sel[0..G).
 * bg_collate (after the host has read n_out = out_node_ptr[G], e_out = out_edge_ptr[G] and allocated):
 *   x [n_out, F], edge_index [2, e_out] (+ the slot's node offset), edge_attr [e_out, Fe], batch [n_out], y [G].
 * An 80 k-graph inference set (~90 GB) fits the 180 GB of a B200: no host collate, no PCIe traffic per batch. */
/* bg_expand_wire: the compact host->device wire format of an inference batch (buckgnn_b200/pipeline.py: WireBatch) ->
 * the PyG tensors `BuckGNN.forward(x, edge_index, edge_attr, batch)` takes (INFERENCE.py:135-136).  wire_edges
 * [2, E_wire] int32 holds every graph's explicit edges (global node ids, graph g at wire_ptr[g]..wire_ptr[g+1]); a graph
 * with full_ptr[g+1] - full_ptr[g] > its explicit count has an IMPLICIT super node = its last node: the hub pairs
 * (s, i), (i, s), i ascending, are appended after its explicit edges, the order `create_super_node` emits
 * (Dataset_Preparation/VirtualEdgeCreate.py:106-111).  Writes edge_index [2, E_full] int64 and batch [N] int64.
 * node_ptr / wire_ptr / full_ptr: DEVICE [G+1] int64. */
int bg_expand_wire(const int32_t* wire_edges, int64_t e_wire, const int64_t* node_ptr, const int64_t* wire_ptr,
                   const int64_t* full_ptr, int64_t n_graphs, int64_t e_full, int64_t* edge_index, int64_t* batch,
                   void* stream);
int bg_collate_ptr(const int64_t* sel, int64_t n_graphs, const int64_t* node_ptr, const int64_t* edge_ptr,
                   int64_t* out_node_ptr, int64_t* out_edge_ptr, void* stream);
int bg_collate(const float* x_all, int32_t n_features, const int64_t* ei_all, int64_t e_all, const float* ea_all,
               int32_t n_edge_features, const float* y_all, const int64_t* sel, int64_t n_graphs,
               const int64_t* node_ptr, const int64_t* edge_ptr, const int64_t* out_node_ptr,
               const int64_t* out_edge_ptr, int64_t n_out, int64_t e_out,
               float* x, int64_t* edge_index, float* edge_attr, int64_t* batch, float* y, void* stream);
/* Loss + metric epilogue of the eigenvalue head, replacing per batch `criterion(normalizer.denormalize_eigenvalue(pred),
 * normalizer.denormalize_eigenvalue(batch.y))` + `MAPE_error(pred, batch.y, "buckling", normalizer).item()`
 * (TRAIN_FINAL.py:262-263, 340-341; Normalizer.py:207-215, Utils/Losses.py:755-761, Metrics.py:4-12):
 *   pd = pred*scale + center, td = y*scale + center;  out2[0] = mean(|pd-td| / (|td|+eps));  out2[1] = 100*mean(|td-pd|/|td|)
 *   dpred (nullable, [G]) = d out2[0] / d pred;  accum3 (nullable) += {loss, mape, 1} (epoch sums without host syncs). */
int bg_eigen_loss(const float* pred, const float* y, int64_t n_graphs, float scale, float center, float eps,
                  float* out2, float* dpred, float* accum3, void* stream);
/* keep[r*512 + c] = 1 if dropout keeps element (r, c) for (seed, dropout_p) -- lets a test apply the same mask. */
int bg_dropout_mask(uint64_t seed, float dropout_p, int64_t n_rows, uint8_t* keep, void* stream);

/* ------------------------------------------------------------------ helpers
 * fp32 -> bf16 / f16 (round to nearest even) cast of a contiguous buffer (weight packing). */
int bg_cast_f32(const float* src, void* dst, int dst_dtype, int64_t n, void* stream);
/* hi/lo split for the 3xTF32 "fp32-GEMM" mode: hi = src with the low 13 mantissa bits
 * cleared (exactly representable in tf32), lo = src - hi.  hi may be NULL: tcgen05 kind::tf32 ignores the low 13
 * mantissa bits of an fp32 operand (verified bit-for-bit on B200, tools/tf32_trunc_probe.py), so `src` itself
 * serves as the hi operand and only lo needs to be materialised. */
int bg_split_tf32(const float* src, float* hi, float* lo, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BUCKGNN_B200_H_ */
