"""The BuckGNN forward as a sequence of C-ABI calls on the current CUDA stream.

torch is used here for device memory (caching allocator), streams and nothing else:
every arithmetic step of the hot path is one of the hand-written kernels behind
include/buckgnn_b200.h.  There is no fallback: a CPU tensor or a missing library
raises.

Reference path restated (Models/BuckGNN.py):
  :323      node_encoder            -> bg_encoder_front + bg_gemm512 (128 -> 512)
  :445-458  GraphSAGE layer loop    -> per layer bg_sage_aggregate + bg_gemm512 with the
                                       fused bias / L2-normalize / BN / ReLU / skip epilogue
  :274,515  global_mean_pool+decoder-> bg_pool_head
The CSR (bg_csr_build) and graph offsets (bg_graph_ptr_build) are rebuilt from the raw
`edge_index` / `batch` on every call unless the caller opts into `cache_index`.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import capi

# precision mode -> (activation storage, weight storage) of the tensor-core GEMMs
#   fp16  : fp16 x fp16, fp32 accumulate.  11-bit significands: the rounding of the SHARED
#           weights (the error that does not average out over nodes) is 8x smaller than
#           with bf16, at the same cost.  Activations must stay below 65504, which the
#           L2-normalise + BN of every layer guarantees for mean / max aggregation.
#   bf16  : bf16 x bf16 (fp32-like range, ~1e-3 systematic error on the prediction)
#   tf32  : fp32 storage, operands read as tf32 (default for sum/add aggregation, whose
#           hub rows sum thousands of terms and can leave the fp16 range)
#   fp32  : fp32 storage, hi/lo split operands, 3 tf32 products per term ("fp32-GEMM mode")
# (tcgen05 kind::f16 rejects A = bf16 with B = fp16 -- illegal instruction on sm_100a --
#  so there is no mixed mode.)
_TORCH = {capi.BG_BF16: torch.bfloat16, capi.BG_F16: torch.float16, capi.BG_F32: torch.float32}
PRECISION_FORMATS = {
    "fp16": (capi.BG_F16, capi.BG_F16),
    "bf16": (capi.BG_BF16, capi.BG_BF16),
    "tf32": (capi.BG_F32, capi.BG_F32),
    "fp32": (capi.BG_F32, capi.BG_F32),
}
PRECISIONS = tuple(PRECISION_FORMATS)


def default_precision(aggr: str) -> str:
    return "fp16" if aggr in ("mean", "max") else "tf32"


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class _KernelTimers:
    """Optional CUDA-event brackets around each kernel class, recorded on the launching
    stream (bench.py turns them on for its timed region; off by default = zero cost).
    With BUCKGNN_NVTX=1 in the environment (or `TIMERS.nvtx = True`) every span also opens an NVTX range
    of the same name, so an `ncu --nvtx --nvtx-include "sage_update/"` capture or a timeline groups the
    launches by what they do (tools/profile.sh)."""

    def __init__(self):
        self.enabled = False
        self.nvtx = os.environ.get("BUCKGNN_NVTX", "0") not in ("", "0")
        self.spans = []

    def enable(self):
        self.enabled, self.spans = True, []

    def disable(self):
        self.enabled, self.spans = False, []

    class _Span:
        def __init__(self, owner, name):
            self.owner, self.name = owner, name

        def __enter__(self):
            self.pushed = self.owner.nvtx
            if self.pushed:
                torch.cuda.nvtx.range_push(self.name)
            if self.owner.enabled:
                self.e0 = torch.cuda.Event(enable_timing=True)
                self.e1 = torch.cuda.Event(enable_timing=True)
                self.e0.record()
            return self

        def __exit__(self, *a):
            if self.owner.enabled:
                self.e1.record()
                self.owner.spans.append((self.name, self.e0, self.e1))
            if self.pushed:
                torch.cuda.nvtx.range_pop()

    def span(self, name):
        return self._Span(self, name)

    def summary(self):
        """{name: (total_ms, calls)} -- synchronises."""
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.spans:
            ms, n = out.get(name, (0.0, 0))
            out[name] = (ms + e0.elapsed_time(e1), n + 1)
        return out


TIMERS = _KernelTimers()


def LAUNCHES_PER_FORWARD(num_layers: int, folded: bool = True, fused_pool: bool = False) -> int:
    """Kernels of ours launched by one GraphSAGE forward: CSR build 7 (hist, 3 scan, fill,
    2 sorts) + batch_info + publish_words + graph_ptr + encoder front 1 (+ encoder GEMM when layer 0 is not folded;
    + row indicator when it is) + per layer (aggregate rows + hubs + GEMM) + pool 2 (+ the block-flag kernel of a pool-fused last layer).
    (memsets and the 16-byte info read-back are not counted.)"""
    extra = 1 if fused_pool else 0      # bg_pool_block_flags
    if folded:                          # (the row-indicator kernel is skipped when no node is isolated)
        return 7 + 3 + 1 + 3 * num_layers + 2 + extra
    return 7 + 3 + 2 + 3 * num_layers + 2 + extra


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"buckgnn_b200: `{name}` must be a CUDA tensor (got {t.device}); the hot path has "
                           "no CPU implementation")


@dataclass
class GraphIndex:
    """CSR of the batch keyed by target node + per-graph node offsets (all int32, on device)."""
    n_nodes: int
    n_edges: int
    rowptr: torch.Tensor
    col: torch.Tensor
    perm: torch.Tensor
    big_rows: torch.Tensor
    n_big: int
    graph_ptr: torch.Tensor
    n_graphs: int
    # "range hubs" (bg_csr_build): set when EVERY big row's neighbour list is a contiguous run of rows --
    # the reference's super node -- so bg_sage_aggregate can fold the hub rows into its row pass
    hub_lo: Optional[torch.Tensor] = None
    hub_of_row: Optional[torch.Tensor] = None
    hub_max_degree: int = 0
    has_empty_rows: bool = True          # some node has no CSR entries (bg_csr_build info[6])


class PendingGraphIndex:
    """K1 in flight.  `begin_graph_index` enqueues the CSR build (and the `batch` scan) on the
    current stream and publishes the result words (error flag, hub-row count, graph count,
    sortedness, hub ranges) to pinned host memory; `finish()` blocks only on the event behind that
    -- kernels the caller enqueued in between (the node encoder) keep the GPU busy meanwhile.  This is the one
    host<->device sync of a forward, the same kind PyG's `batch.max()+1` does."""

    def __init__(self, edge_index, batch, n_nodes, key_row):
        _require_cuda(edge_index, "edge_index")
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise ValueError("edge_index must be an int64 tensor of shape [2, E]")
        self.edge_index = edge_index.contiguous()
        dev = edge_index.device
        self.E, self.N = edge_index.shape[1], int(n_nodes)
        E, N = self.E, self.N
        s = _stream()
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(N + 1, **i32)
        self.col = torch.empty(max(E, 1), **i32)
        self.perm = torch.empty(max(E, 1), **i32)
        self.big_rows = torch.empty(capi.csr_max_big_rows(E), **i32)
        self.hub_lo = torch.empty(capi.csr_max_big_rows(E), **i32)
        self.hub_of_row = torch.empty(max(N, 1), **i32)
        self.info = torch.zeros(8, **i32)
        ws_bytes = capi.csr_workspace_bytes(N, E)
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with TIMERS.span("csr_build"):
            capi.csr_build(self.edge_index.data_ptr(), E, N, key_row, self.rowptr.data_ptr(), self.col.data_ptr(),
                           self.perm.data_ptr(), self.big_rows.data_ptr(), self.info.data_ptr(),
                           self._ws.data_ptr(), ws_bytes, s, hub_lo=self.hub_lo.data_ptr(),
                           hub_of_row=self.hub_of_row.data_ptr())
        self.batch = None
        if batch is not None:
            _require_cuda(batch, "batch")
            if batch.dtype != torch.int64 or batch.dim() != 1 or batch.shape[0] != N:
                raise ValueError("batch must be an int64 tensor of shape [N]")
            self.batch = batch.contiguous()
            capi.batch_info(self.batch.data_ptr(), N, self.info[2:].data_ptr(), s)
        # result words -> pinned host memory by SM stores (bg_publish_words), then an event on THIS stream: no
        # copy engine involved, so the read-back cannot queue behind the H2D transfer of the next batch
        self._host = torch.zeros(8, dtype=torch.int32).pin_memory()
        capi.publish_words(self.info.data_ptr(), self._host.data_ptr(), 8, s)
        self._done = torch.cuda.Event()
        self._done.record()

    def finish(self) -> "GraphIndex":
        self._done.synchronize()                      # the one sync of the forward
        host = self._host.tolist()
        N, E = self.N, self.E
        i32 = dict(dtype=torch.int32, device=self.edge_index.device)
        if host[0] & 1:
            raise IndexError("edge_index contains node ids outside [0, num_nodes)")
        n_big = host[1]
        if self.batch is None:
            n_graphs = 1
            graph_ptr = torch.tensor([0, N], **i32)
        else:
            if host[3]:
                raise ValueError("buckgnn_b200 needs a sorted, non-negative `batch` vector (PyG DataLoader order)")
            n_graphs = host[2] if N > 0 else 0
            graph_ptr = torch.empty(n_graphs + 1, **i32)
            capi.graph_ptr_build(self.batch.data_ptr(), N, n_graphs, graph_ptr.data_ptr(), _stream())
        ranges = n_big > 0 and host[4] == 0
        return GraphIndex(N, E, self.rowptr, self.col, self.perm, self.big_rows, n_big, graph_ptr, n_graphs,
                          hub_lo=self.hub_lo if ranges else None, hub_of_row=self.hub_of_row if ranges else None,
                          hub_max_degree=host[5] if ranges else 0, has_empty_rows=bool(host[6]) or N == 0)


def begin_graph_index(edge_index: torch.Tensor, batch: Optional[torch.Tensor], n_nodes: int,
                      key_row: int = 1) -> PendingGraphIndex:
    return PendingGraphIndex(edge_index, batch, n_nodes, key_row)


def build_graph_index(edge_index: torch.Tensor, batch: Optional[torch.Tensor], n_nodes: int,
                      key_row: int = 1) -> GraphIndex:
    """K1, blocking form."""
    return begin_graph_index(edge_index, batch, n_nodes, key_row).finish()


# ----------------------------------------------------------------------------- packed weights
@dataclass
class LinearPack:
    """A weight [512, K] (nn.Linear layout) in the operand format of one precision mode."""
    k: int
    parts: Tuple[torch.Tensor, ...]     # 16-bit / tf32: (w,)   fp32: (w_hi, w_lo)
    code: int = capi.BG_F32             # bg_dtype of the parts


def pack_linear(weight: torch.Tensor, precision: str) -> LinearPack:
    w = weight.detach().to(torch.float32).contiguous()
    k = w.shape[1]
    s = _stream()
    code = PRECISION_FORMATS[precision][1]
    if code != capi.BG_F32:
        out = torch.empty(w.shape, dtype=_TORCH[code], device=w.device)
        capi.cast_f32(w.data_ptr(), out.data_ptr(), code, w.numel(), s)
        return LinearPack(k, (out,), code)
    if precision == "tf32":
        return LinearPack(k, (w.clone(),), code)
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    capi.split_tf32(w.data_ptr(), hi.data_ptr(), lo.data_ptr(), w.numel(), s)
    return LinearPack(k, (hi, lo), code)


@dataclass
class SageLayerPack:
    lin_l: LinearPack
    lin_r: LinearPack
    bias: torch.Tensor                   # f32 [512], HOST (travels in the kernel parameters)
    bn_scale: Optional[torch.Tensor]     # f32 [512], HOST   gamma / sqrt(var + eps)
    bn_shift: Optional[torch.Tensor]     # f32 [512], HOST   beta - mean * scale


def fold_batchnorm(bn: torch.nn.BatchNorm1d) -> Tuple[torch.Tensor, torch.Tensor]:
    """Eval-mode BatchNorm1d as one multiply-add per column (Models/BuckGNN.py:451)."""
    scale = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps))
    shift = (bn.bias.detach().float() - bn.running_mean.detach().float() * scale)
    return scale.cpu().contiguous(), shift.cpu().contiguous()


def host_vector(t: torch.Tensor) -> torch.Tensor:
    """fp32 host copy of a [512] epilogue vector (bias / BN scale / BN shift)."""
    return t.detach().float().cpu().contiguous()


class Activation:
    """An [N, 512] (or [N, K]) activation in the operand format of a precision mode."""

    def __init__(self, n: int, width: int, precision: str, device):
        self.precision = precision
        self.code = PRECISION_FORMATS[precision][0]
        self.dtype = _TORCH[self.code]
        self.data = torch.empty((n, width), dtype=self.dtype, device=device)
        self.hi = self.lo = None
        if precision == "fp32":
            # tcgen05 kind::tf32 reads the upper 19 bits of an fp32 operand (truncation, verified bit-for-bit by
            # tools/tf32_trunc_probe.py), so the data itself IS the hi operand; only lo = x - trunc(x) is stored
            self.hi = self.data
            self.lo = torch.empty_like(self.data)

    def refresh_split(self):
        if self.precision == "fp32":
            capi.split_tf32(self.data.data_ptr(), None, self.lo.data_ptr(), self.data.numel(), _stream())


def _segments(act: Activation, w: LinearPack):
    """K-segments of act . w^T for the mode: 1, or 3 for fp32 (3xTF32: hi*hi + hi*lo + lo*hi)."""
    k = w.k
    ld = act.data.shape[1]
    if act.precision != "fp32":
        return [(act.data.data_ptr(), ld, w.parts[0].data_ptr(), k, k)]
    w_hi, w_lo = w.parts
    return [(act.hi.data_ptr(), ld, w_hi.data_ptr(), k, k),
            (act.hi.data_ptr(), ld, w_lo.data_ptr(), k, k),
            (act.lo.data_ptr(), ld, w_hi.data_ptr(), k, k)]


def gemm512(segs, m: int, precision: str, out: Activation, *, cta_group: int = 2, **epi) -> None:
    a_code, b_code = PRECISION_FORMATS[precision]
    capi.gemm512(segs, m, a_code, b_code, out.data.data_ptr(), out.code, out.data.shape[1], _stream(),
                 cta_group=cta_group, **epi)
    out.refresh_split()


def gemm(segs, m: int, precision: str, out: Activation, *, cta_group: int = 2, **epi) -> None:
    """The update GEMM for the width of `out`: bg_gemm128 for 128-wide rows (a hidden_channels = 128 model on its own
    kernels; bg_gemm128_gathered when there are gathered addends), else bg_gemm512."""
    if out.data.shape[1] != 128:
        return gemm512(segs, m, precision, out, cta_group=cta_group, **epi)
    a_code, b_code = PRECISION_FORMATS[precision]
    fn = capi.gemm128_gathered if epi.get("gather") else capi.gemm128
    fn(segs, m, a_code, b_code, out.data.data_ptr(), out.code, out.data.shape[1], _stream(),
       cta_group=cta_group, **epi)
    out.refresh_split()


def aggregate(x: Activation, out: Activation, idx: GraphIndex, aggr: str, fold_hubs: bool = True) -> None:
    """K2 over [N,512] rows, or [N,128] rows (the encoder hidden layer of the folded first layer)."""
    width = x.data.shape[1]
    ws_bytes = capi.aggregate_workspace_bytes(idx.n_big)
    hub = {}
    if fold_hubs and idx.hub_lo is not None and width == 512 and aggr != "max":
        fold_bytes = capi.hubfold_workspace_bytes(idx.n_nodes, x.code, idx.n_big, idx.hub_max_degree)
        # the per-(hub, band, warp) partials are written and read once: only worth it while they stay
        # small next to the pass over x they replace (many tiny hubs -> generic hub kernel)
        if fold_bytes <= x.data.numel() * x.data.element_size() // 4 + (1 << 20):
            ws_bytes = fold_bytes
            hub = dict(hub_lo=idx.hub_lo.data_ptr(), hub_of_row=idx.hub_of_row.data_ptr(),
                       hub_max_degree=idx.hub_max_degree)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.data.device)
    with TIMERS.span("aggregate" if width == 512 else "aggregate128"):
        capi.sage_aggregate(x.data.data_ptr(), out.data.data_ptr(), x.code, idx.n_nodes, idx.rowptr.data_ptr(),
                            idx.col.data_ptr(), idx.big_rows.data_ptr(), idx.n_big, capi.AGGR_CODES[aggr],
                            ws.data_ptr(), ws_bytes, _stream(), width=width, **hub)
    out.refresh_split()


def encoder_hidden(x: torch.Tensor, enc_w: Dict[str, torch.Tensor], precision: str,
                   row_gather: Optional[torch.Tensor] = None, nonfinite: Optional[torch.Tensor] = None) -> "Activation":
    """First two Linear+ReLU of an encoder -> [n,128] activation (K5 front).  `nonfinite` (int32 [1], device) is
    raised when the 16-bit storage format cannot hold a value of the (un-normalised) hidden layer."""
    f = x.shape[1]
    n = x.shape[0] if row_gather is None else row_gather.shape[0]
    h = Activation(n, 128, precision, x.device)
    with TIMERS.span("encoder_front"):
        capi.encoder_front(x.data_ptr(), n, f, enc_w["w1"].data_ptr(), enc_w["b1"].data_ptr(),
                           enc_w["w2"].data_ptr(), enc_w["b2"].data_ptr(), h.data.data_ptr(), h.code, _stream(),
                           row_gather=_p(row_gather), nonfinite=_p(nonfinite))
    h.refresh_split()
    return h


@dataclass
class FoldedLayer0Pack:
    """SAGE layer 0 with the encoder's last Linear folded in (exact algebra; the encoder output
    x0 = h W3^T + b3 is never materialised):
        mean_j(x0_j) W_l^T + x0_i W_r^T + b_l
      = mean_j(h_j) (W_l W3)^T + h_i (W_r W3)^T + [deg_i > 0] (W_l b3) + (W_r b3 + b_l)
    (for sum/add aggregation the indicator is deg_i).  K = 128 + 128 + 64 instead of 1024, and the
    aggregation moves 128 instead of 512 columns."""
    wl3: LinearPack
    wr3: LinearPack
    wgate: LinearPack
    bias: torch.Tensor                   # HOST f32 [512]
    bn_scale: Optional[torch.Tensor]
    bn_shift: Optional[torch.Tensor]
    as_count: bool
    bias_all_gated: Optional[torch.Tensor] = None   # HOST f32 [512]: bias + W_l b3, valid when every row's gate is 1


def pack_folded_layer0(enc_last: torch.nn.Linear, conv, bn, aggr: str, precision: str,
                       width: int = 512) -> Optional[FoldedLayer0Pack]:
    """`width`: the layer's output width (512, or 128 for a hidden_channels = 128 model, whose encoder's last Linear
    reads the 64-wide hidden layer stored 128 wide: W3 is zero-padded to 128 columns).
    None when a folded weight does not fit its operand format (fp16 with sum / add aggregation: the degree digits'
    gate columns carry W_l b3 x 65536, inf once |W_l b3| > ~1, and the MMA would make every row 0 x inf = NaN); the
    caller then runs layer 0 unfolded."""
    dev = conv.lin_l.weight.device
    d64 = lambda t: t.detach().to(torch.float64).cpu()
    W3, b3 = d64(enc_last.weight), d64(enc_last.bias)
    W3 = torch.nn.functional.pad(W3, (0, 128 - W3.shape[1]))
    Wl, bl, Wr = d64(conv.lin_l.weight), d64(conv.lin_l.bias), d64(conv.lin_r.weight)
    lp = lambda w: pack_linear(w.to(torch.float32).to(dev), precision)
    gate = torch.cat([(Wl @ b3)[:, None], torch.zeros(width, 63, dtype=torch.float64)], 1)
    if aggr in ("sum", "add"):
        # the A operand carries deg_i as three base-256 digits (bg_expand_rowptr as_count): a super node's degree
        # (thousands) is not exact in 8 / 11 significant bits, its digits are
        gate[:, 1] = gate[:, 0] * 256.0
        gate[:, 2] = gate[:, 0] * 65536.0
    wl3, wr3, wgate = lp(Wl @ W3), lp(Wr @ W3), lp(gate)
    if not all(bool(torch.isfinite(t).all()) for pk in (wl3, wr3, wgate) for t in pk.parts):
        return None
    scale, shift = fold_batchnorm(bn) if bn is not None else (None, None)
    return FoldedLayer0Pack(wl3, wr3, wgate, (Wr @ b3 + bl).to(torch.float32).contiguous(),
                            scale, shift, aggr in ("sum", "add"),
                            bias_all_gated=(Wr @ b3 + bl + Wl @ b3).to(torch.float32).contiguous())


def sage_layer0_folded(h: "Activation", out: "Activation", idx: GraphIndex, w: FoldedLayer0Pack, *, aggr: str,
                       normalize: bool, relu: bool, cta_group: int = 2) -> None:
    n = idx.n_nodes
    mh = Activation(n, 128, h.precision, h.data.device)
    aggregate(h, mh, idx, aggr)
    segs = _segments(mh, w.wl3) + _segments(h, w.wr3)
    bias = w.bias
    if not w.as_count and not idx.has_empty_rows:
        bias = w.bias_all_gated          # mean aggregation, every node has a neighbour: the gate is 1 on every row
    else:
        ind = Activation(n, 64, h.precision, h.data.device)
        capi.expand_rowptr(idx.rowptr.data_ptr(), n, idx.n_edges, None, None, ind.data.data_ptr(), ind.code, _stream(),
                           as_count=w.as_count)
        ind.refresh_split()
        # indicator / degree digits are exact in tf32 (lo part 0): of the 3xTF32 products only hi*w_hi + hi*w_lo remain
        segs = segs + _segments(ind, w.wgate)[:2]
    with TIMERS.span("sage_update0"):
        gemm(segs, n, h.precision, out, cta_group=cta_group, bias=bias.data_ptr(), bn_scale=_p(w.bn_scale),
             bn_shift=_p(w.bn_shift), normalize=normalize, relu=relu)


def pack_encoder(enc, precision: str, width: int = 512) -> Tuple[Dict[str, torch.Tensor], LinearPack]:
    """(enc_w, w3) of `encoder_forward` for a node / edge encoder.  `width` 128: the 2-layer encoder Linear(F,64) ReLU
    Linear(64,128) of h <= 128 (Models/BuckGNN.py:41-48) runs on the same kernels by exact embedding: [I; 0] as the
    second Linear (the 64-wide hidden layer stored 128 wide), then Linear(64,128) with W zero-padded to [128, 128]."""
    f32 = lambda t: t.detach().float().contiguous()
    enc_w = {"w1": f32(enc[0].weight), "b1": f32(enc[0].bias)}
    if width == 512:
        enc_w.update(w2=f32(enc[2].weight), b2=f32(enc[2].bias), b3_host=host_vector(enc[4].bias))
        return enc_w, pack_linear(enc[4].weight, precision)
    dev = enc[0].weight.device
    w2 = torch.zeros((128, 64), dtype=torch.float32, device=dev)
    w2[:64] = torch.eye(64, device=dev)
    enc_w.update(w2=w2, b2=torch.zeros(128, dtype=torch.float32, device=dev), b3_host=host_vector(enc[2].bias))
    return enc_w, pack_linear(torch.nn.functional.pad(f32(enc[2].weight), (0, 64)), precision)


def encoder_forward(x: torch.Tensor, enc_w: Dict[str, torch.Tensor], w3: LinearPack, precision: str,
                    out: Activation, cta_group: int, row_gather: Optional[torch.Tensor] = None,
                    nonfinite: Optional[torch.Tensor] = None) -> None:
    """node_encoder / edge_encoder (Models/BuckGNN.py:68-82): two fp32 CUDA-core layers, then 128->512 on
    tcgen05.  `row_gather` [n] int32 reads input row row_gather[i] for output row i."""
    h = encoder_hidden(x, enc_w, precision, row_gather, nonfinite)
    n = h.data.shape[0]
    with TIMERS.span("encoder_gemm"):
        gemm(_segments(h, w3), n, precision, out, cta_group=cta_group, bias=enc_w["b3_host"].data_ptr())


@dataclass
class PoolBlocks:
    """What a pool-fused last layer hands to `pool_head`: fp32 column sums of every 32-row block of the layer's
    output, and the flags of the blocks whose rows were stored as well (first / last row of a graph)."""
    sums: torch.Tensor       # [ceil(N/32), width] f32
    keep: torch.Tensor       # [ceil(N/32)] uint8


def new_pool_blocks(idx: GraphIndex, device, width: int = 512) -> PoolBlocks:
    nb = (idx.n_nodes + 31) // 32
    keep = torch.empty(max(nb, 1), dtype=torch.uint8, device=device)
    capi.pool_block_flags(idx.graph_ptr.data_ptr(), idx.n_graphs, idx.n_nodes, keep.data_ptr(), _stream())
    return PoolBlocks(torch.empty((max(nb, 1), width), dtype=torch.float32, device=device), keep)


def can_fuse_pool(precision: str, normalize: bool, residual: bool) -> bool:
    """The pool-fused epilogue exists for the 16-bit normalize epilogue without addends (the last SAGE layer)."""
    return PRECISION_FORMATS[precision][0] != capi.BG_F32 and normalize and not residual


# The fused SAGE layer (bg_sage_fused512: the aggregate operand is gathered inside the GEMM kernel and never written to
# global memory).  Opt-in: BUCKGNN_FUSE_AGGREGATE=1 in the environment, or `model.fuse_aggregate = True`.
FUSE_AGGREGATE_DEFAULT = os.environ.get("BUCKGNN_FUSE_AGGREGATE", "0") not in ("", "0")


def can_fuse_aggregate(precision: str, aggr: str, normalize: bool) -> bool:
    return precision in ("fp16", "bf16") and aggr in ("mean", "sum", "add") and normalize


def sage_layer_fused(x: Activation, out: Activation, idx: GraphIndex, layer: SageLayerPack, *, aggr: str, relu: bool,
                     residual: bool, pool_blocks: Optional[PoolBlocks] = None) -> None:
    """One reference layer iteration (Models/BuckGNN.py:447-457) as ONE kernel (+ the hub rows' aggregates, one small
    launch over the few super-node rows): mean / sum aggregation, lin_l / lin_r, F.normalize, BatchNorm, ReLU, skip."""
    dev = x.data.device
    hub_agg = None
    if idx.n_big > 0:
        hub_agg = torch.empty((idx.n_big, 512), dtype=x.data.dtype, device=dev)
        ws_bytes = capi.aggregate_workspace_bytes(idx.n_big)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with TIMERS.span("aggregate_hubs"):
            capi.sage_aggregate_hubs(x.data.data_ptr(), x.code, idx.rowptr.data_ptr(), idx.col.data_ptr(),
                                     idx.big_rows.data_ptr(), idx.n_big, capi.AGGR_CODES[aggr], hub_agg.data_ptr(),
                                     ws.data_ptr(), ws_bytes, _stream())
    k = layer.lin_l.k
    segs = [(None, 0, layer.lin_l.parts[0].data_ptr(), k, k)] + _segments(x, layer.lin_r)
    pool = {} if pool_blocks is None else dict(pool_block_sums=pool_blocks.sums.data_ptr(),
                                               pool_block_keep=pool_blocks.keep.data_ptr())
    a_code, b_code = PRECISION_FORMATS[x.precision]
    with TIMERS.span("sage_fused" if pool_blocks is None else "sage_fused_pool"):
        capi.sage_fused512(segs, idx.n_nodes, a_code, b_code, out.data.data_ptr(), out.code, out.data.shape[1], _stream(),
                           x=x.data.data_ptr(), ldx=x.data.shape[1], rowptr=idx.rowptr.data_ptr(), col=idx.col.data_ptr(),
                           aggr=capi.AGGR_CODES[aggr], hub_agg=_p(hub_agg), big_rows=idx.big_rows.data_ptr(), n_big=idx.n_big,
                           bias=layer.bias.data_ptr(), bn_scale=_p(layer.bn_scale), bn_shift=_p(layer.bn_shift),
                           residual=x.data.data_ptr() if residual else None, ldr=x.data.shape[1], relu=relu, **pool)
    out.refresh_split()


def sage_layer(x: Activation, agg: Activation, out: Activation, idx: GraphIndex, layer: SageLayerPack, *,
               aggr: str, normalize: bool, relu: bool, residual: bool, cta_group: int,
               pool_blocks: Optional[PoolBlocks] = None, fuse_aggregate: bool = False) -> None:
    """One reference layer iteration (Models/BuckGNN.py:447-457) = aggregate + fused update GEMM.
    `pool_blocks` (last layer of a graph-level model): the epilogue sums the output rows per 32-row block for
    `pool_head` instead of storing them (only the blocks at graph boundaries are stored)."""
    if fuse_aggregate and can_fuse_aggregate(x.precision, aggr, normalize):
        return sage_layer_fused(x, out, idx, layer, aggr=aggr, relu=relu, residual=residual, pool_blocks=pool_blocks)
    aggregate(x, agg, idx, aggr)
    segs = _segments(agg, layer.lin_l) + _segments(x, layer.lin_r)
    pool = {} if pool_blocks is None else dict(pool_block_sums=pool_blocks.sums.data_ptr(),
                                               pool_block_keep=pool_blocks.keep.data_ptr())
    with TIMERS.span("sage_update" if pool_blocks is None else "sage_update_pool"):
        gemm(segs, idx.n_nodes, x.precision, out, cta_group=cta_group,
                bias=layer.bias.data_ptr(), bn_scale=_p(layer.bn_scale), bn_shift=_p(layer.bn_shift),
                residual=x.data.data_ptr() if residual else None, ldr=x.data.shape[1],
                normalize=normalize, relu=relu, **pool)


def pack_decoder(dec, width: int = 512) -> Dict[str, torch.Tensor]:
    """The fp32 decoder weights w1, b1, w2, b2, w3, b3 of `pool_head`.  `width` 128: the 2-layer decoder
    Linear(in,64) ReLU Linear(64,out) of h <= 128 (Models/BuckGNN.py:41-65) in the 3-layer form bg_pool_head128
    takes (include/buckgnn_b200.h): w1 = [W1; 0], w2 = [I64 | 0], w3 = W2."""
    f32 = lambda t: t.detach().float().contiguous()
    if width == 512:
        return {"w1": f32(dec[0].weight), "b1": f32(dec[0].bias), "w2": f32(dec[2].weight),
                "b2": f32(dec[2].bias), "w3": f32(dec[4].weight), "b3": f32(dec[4].bias)}
    dev = dec[0].weight.device
    w1 = torch.zeros((128, dec[0].in_features), dtype=torch.float32, device=dev)
    b1 = torch.zeros(128, dtype=torch.float32, device=dev)
    w1[:64], b1[:64] = f32(dec[0].weight), f32(dec[0].bias)
    w2 = torch.zeros((64, 128), dtype=torch.float32, device=dev)
    w2[:, :64] = torch.eye(64, device=dev)
    return {"w1": w1, "b1": b1, "w2": w2, "b2": torch.zeros(64, dtype=torch.float32, device=dev),
            "w3": f32(dec[2].weight), "b3": f32(dec[2].bias)}


def pool_head(x: Activation, idx: GraphIndex, dec: Dict[str, torch.Tensor], out_dim: int,
              want_pooled: bool = False, pooling: str = "mean", pre: Optional[Dict[str, torch.Tensor]] = None,
              nonfinite: Optional[torch.Tensor] = None, blocks: Optional[PoolBlocks] = None):
    """get_pooling_layer + decoder (Models/BuckGNN.py:246-307, 515-516).  With `blocks` (pool-fused last layer)
    x holds valid rows only in the flagged blocks and the rest comes from the block sums."""
    dev = x.data.device
    g = idx.n_graphs
    mode = capi.POOL_MODES[pooling]
    width = x.data.shape[1]                  # 512, or 128: bg_pool_head128 / bg_pool_head_blocks128
    in_dim = 2 * width if pooling == "supernode_with_pooling" else width
    pred = torch.empty((g, out_dim), dtype=torch.float32, device=dev)
    pooled = torch.empty((g, in_dim), dtype=torch.float32, device=dev) if want_pooled else None
    ws_bytes = capi.pool_workspace_bytes(g)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    head, head_blocks = (capi.pool_head128, capi.pool_head_blocks128) if width == 128 else (capi.pool_head, capi.pool_head_blocks)
    with TIMERS.span("pool_head"):
        if blocks is not None:
            head_blocks(x.data.data_ptr(), x.code, idx.n_nodes, idx.graph_ptr.data_ptr(), g, mode,
                        _p(pre["w"]) if pre else None, _p(pre["b"]) if pre else None,
                        dec["w1"].data_ptr(), dec["b1"].data_ptr(), dec["w2"].data_ptr(), dec["b2"].data_ptr(),
                        dec["w3"].data_ptr(), dec["b3"].data_ptr(), out_dim, pred.data_ptr(), _p(pooled),
                        blocks.sums.data_ptr(), blocks.keep.data_ptr(), ws.data_ptr(), ws_bytes, _stream(),
                        nonfinite=_p(nonfinite))
        else:
            head(x.data.data_ptr(), x.code, idx.n_nodes, idx.graph_ptr.data_ptr(), g, mode,
                 _p(pre["w"]) if pre else None, _p(pre["b"]) if pre else None,
                 dec["w1"].data_ptr(), dec["b1"].data_ptr(), dec["w2"].data_ptr(), dec["b2"].data_ptr(),
                 dec["w3"].data_ptr(), dec["b3"].data_ptr(), out_dim, pred.data_ptr(), _p(pooled),
                 ws.data_ptr(), ws_bytes, _stream(), nonfinite=_p(nonfinite))
    return pred, pooled


def pack_node_head(decoder, precision: str) -> Dict[str, object]:
    """Node-level heads (`decoder(x)` on every node, Models/BuckGNN.py:518-524): the first Linear (512 -> 128)
    runs on the tensor-core GEMM with its weight zero-padded to 512 output rows; the two narrow Linears
    (128 -> 64 -> out) run on bg_sgemm."""
    w1 = decoder[0].weight.detach().float()
    dev = w1.device
    w1p = torch.zeros((512, w1.shape[1]), dtype=torch.float32, device=dev)
    w1p[:w1.shape[0]] = w1
    b1p = torch.zeros(512, dtype=torch.float32)
    b1p[:w1.shape[0]] = decoder[0].bias.detach().float().cpu()
    f32 = lambda t: t.detach().float().contiguous()
    return {"w1": pack_linear(w1p, precision), "b1_host": b1p.contiguous(), "h1_width": w1.shape[0],
            "w2": f32(decoder[2].weight), "b2": f32(decoder[2].bias), "w3": f32(decoder[4].weight), "b3": f32(decoder[4].bias)}


def pack_node_head128(decoder, precision: str) -> Dict[str, torch.Tensor]:
    """The 2-layer decoder Linear(128,64) ReLU Linear(64,out) of h <= 128 (Models/BuckGNN.py:41-65) for
    bg_node_head128: W1 in the operand format of the model's storage format (fp16 / bf16; the exact fp32 weight for the
    fp32-storage modes, whose kernel uses fp32 FMAs), b1, W2 and b2 in fp32."""
    f32 = lambda t: t.detach().float().contiguous()
    w1 = decoder[0].weight
    code = PRECISION_FORMATS[precision][0]
    return {"w1": f32(w1) if code == capi.BG_F32 else pack_linear(w1, precision).parts[0],
            "b1": f32(decoder[0].bias), "w2": f32(decoder[2].weight), "b2": f32(decoder[2].bias)}


def node_head(x: Activation, n: int, head: Dict[str, object], out_dim: int, cta_group: int = 2) -> torch.Tensor:
    """decoder(x) for all n nodes -> [n, out_dim] f32.  128-wide rows (a hidden_channels = 128 model) run on
    bg_node_head128 with `pack_node_head128`'s weights, 512-wide ones on the tensor-core GEMM and bg_sgemm."""
    dev = x.data.device
    s = _stream()
    if x.data.shape[1] == 128:
        out = torch.empty((n, out_dim), dtype=torch.float32, device=dev)
        with TIMERS.span("node_head"):
            capi.node_head128(x.data.data_ptr(), x.code, n, head["w1"].data_ptr(), head["b1"].data_ptr(),
                              head["w2"].data_ptr(), head["b2"].data_ptr(), out_dim, out.data_ptr(), s)
        return out
    h1 = Activation(n, 512, x.precision, dev)
    with TIMERS.span("node_head"):
        gemm512(_segments(x, head["w1"]), n, x.precision, h1, cta_group=cta_group, bias=head["b1_host"].data_ptr(), relu=True)
        k1 = head["h1_width"]
        w2, w3 = head["w2"], head["w3"]
        h2 = torch.empty((n, w2.shape[0]), dtype=torch.float32, device=dev)
        out = torch.empty((n, out_dim), dtype=torch.float32, device=dev)
        for (a, a_code, lda, wt, bias, relu, dst) in ((h1.data, h1.code, 512, w2, head["b2"], True, h2),
                                                     (h2, capi.BG_F32, w2.shape[0], w3, head["b3"], False, out)):
            m_, n_, k_ = n, wt.shape[0], wt.shape[1]
            nb = capi.sgemm_workspace_bytes(m_, n_, k_)
            ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
            capi.sgemm(a.data_ptr(), a_code, lda, 1, wt.data_ptr(), capi.BG_F32, 1, k_, m_, n_, k_, bias.data_ptr(), relu,
                       None, capi.BG_F32, 0, dst.data_ptr(), capi.BG_F32, n_, False, ws.data_ptr(), nb, s)
        assert k1 == w2.shape[1]
    return out


# ----------------------------------------------------------------------------- EA-GNN (GraphNetBlock)
@dataclass
class GNBlockPack:
    """Operand-format weights of one reference `GraphNetBlock` (Models/BuckGNN.py:528-566), split and
    composed so that concatenations never materialise and two Linears fold away:

      edge_mlp L1   cat[x[row], x[col], e] W1^T  =  (x W1a^T)[row] + (x W1b^T)[col] + e W1c^T
      phi L1        cat[x[col], e1] Wp1^T with e1 = h_e W2^T + b2
                    =  (x Wp1a^T)[col] + h_e (Wp1b W2)^T + (Wp1b b2 + bp1)          (edge_mlp L2 folded in)
      scatter_mean then phi L2 then gamma L1 (all linear in between):
                    cat[x, agg] Wg1^T = x Wg1a^T + mean(h_m) (Wg1b Wp2)^T + gate (Wg1b bp2) + bg1
      where gate = 1 for rows with a non-empty scatter_mean segment: a third K = 64 segment whose A operand is
      the indicator matrix from bg_expand_rowptr and whose weight has Wg1b bp2 in column 0.
    """
    w1a: LinearPack; w1b: LinearPack; w1c: LinearPack; b1: torch.Tensor
    w2: LinearPack; b2: torch.Tensor
    wp1a: LinearPack; w3c: LinearPack; b3c: torch.Tensor
    wg1a: LinearPack; wgc: LinearPack; bg1: torch.Tensor; wgate: LinearPack
    wg2: LinearPack; bg2: torch.Tensor
    wb1: LinearPack; bb1: torch.Tensor
    wb2: LinearPack; bb2: torch.Tensor


def pack_gnblock(blk, precision: str, width: int = 512) -> GNBlockPack:
    """`width`: the block's hidden width (512, or 128 for a hidden_channels = 128 model on the 128-wide kernels)."""
    h = width
    dev = blk.edge_mlp[0].weight.device
    d64 = lambda t: t.detach().to(torch.float64).cpu()
    W1, b1 = d64(blk.edge_mlp[0].weight), d64(blk.edge_mlp[0].bias)
    W2, b2 = d64(blk.edge_mlp[2].weight), d64(blk.edge_mlp[2].bias)
    Wp1, bp1 = d64(blk.node_mlp_phi[0].weight), d64(blk.node_mlp_phi[0].bias)
    Wp2, bp2 = d64(blk.node_mlp_phi[2].weight), d64(blk.node_mlp_phi[2].bias)
    Wg1, bg1 = d64(blk.node_mlp_gamma[0].weight), d64(blk.node_mlp_gamma[0].bias)
    Wg2, bg2 = d64(blk.node_mlp_gamma[2].weight), d64(blk.node_mlp_gamma[2].bias)
    Wb1, bb1 = d64(blk.node_mlp_beta[0].weight), d64(blk.node_mlp_beta[0].bias)
    Wb2, bb2 = d64(blk.node_mlp_beta[2].weight), d64(blk.node_mlp_beta[2].bias)
    lp = lambda w: pack_linear(w.to(torch.float32).to(dev), precision)
    hv = lambda b: b.to(torch.float32).contiguous()
    Wp1b, Wg1b = Wp1[:, h:], Wg1[:, h:]
    return GNBlockPack(
        w1a=lp(W1[:, :h]), w1b=lp(W1[:, h:2 * h]), w1c=lp(W1[:, 2 * h:]), b1=hv(b1),
        w2=lp(W2), b2=hv(b2),
        wp1a=lp(Wp1[:, :h]), w3c=lp(Wp1b @ W2), b3c=hv(Wp1b @ b2 + bp1),
        wg1a=lp(Wg1[:, :h]), wgc=lp(Wg1b @ Wp2), bg1=hv(bg1),
        wgate=lp(torch.cat([(Wg1b @ bp2)[:, None], torch.zeros(h, 63, dtype=torch.float64)], 1)),
        wg2=lp(Wg2), bg2=hv(bg2), wb1=lp(Wb1), bb1=hv(bb1), wb2=lp(Wb2), bb2=hv(bb2))


@dataclass
class EdgeIndexExtras:
    row_of: torch.Tensor     # [E] int32: key node of CSR slot i
    iota: torch.Tensor       # [E] int32: 0..E-1
    nonempty: "Activation"   # [N, 64]: column 0 = 1 where the node has >= 1 CSR slot


def edge_extras(idx: GraphIndex, precision: str) -> EdgeIndexExtras:
    dev = idx.rowptr.device
    e = max(idx.n_edges, 1)
    row_of = torch.empty(e, dtype=torch.int32, device=dev)
    iota = torch.empty(e, dtype=torch.int32, device=dev)
    nonempty = Activation(idx.n_nodes, 64, precision, dev)
    capi.expand_rowptr(idx.rowptr.data_ptr(), idx.n_nodes, idx.n_edges, row_of.data_ptr(), iota.data_ptr(),
                       nonempty.data.data_ptr(), nonempty.code, _stream())
    nonempty.refresh_split()
    return EdgeIndexExtras(row_of, iota, nonempty)


def add_into(out: Activation, a: Activation, b: Activation) -> None:
    capi.add(a.data.data_ptr(), b.data.data_ptr(), None, out.data.data_ptr(), out.code, out.data.numel(), _stream())
    out.refresh_split()


class GNBlockBuffers:
    """Scratch activations of the EA-GNN layer loop (allocated once per forward)."""

    def __init__(self, n: int, e: int, precision: str, device, width: int = 512):
        mk = lambda rows: Activation(rows, width, precision, device)
        self.P, self.Q, self.R, self.mh, self.g1, self.xg, self.t, self.s, self.x_alt = (mk(n) for _ in range(9))
        self.he, self.hm, self.e_alt = (mk(max(e, 1)) for _ in range(3))


def gnblock_layer(x: Activation, e: Activation, buf: GNBlockBuffers, idx: GraphIndex, ex: EdgeIndexExtras,
                  w: GNBlockPack, *, skip: bool, need_edges_out: bool, cta_group: int = 2):
    """One iteration of the EA-GNN loop (Models/BuckGNN.py:378-387): returns (x_next, e_next).
    Edge tensors live in CSR order keyed by `row = edge_index[0]` (idx built with key_row=0), so
    scatter_mean(messages, row) is a segmented mean over contiguous slots.  The row width (512, or 128 for a
    hidden_channels = 128 model) is that of `x`; `gemm` picks the kernel for it."""
    prec, n, ne = x.precision, idx.n_nodes, idx.n_edges
    width = x.data.shape[1]
    hp = lambda t: t.data_ptr()
    G = lambda out, segs, m, **kw: gemm(segs, m, prec, out, cta_group=cta_group, **kw)
    with TIMERS.span("gn_node_gemms"):
        G(buf.P, _segments(x, w.w1a), n)
        G(buf.Q, _segments(x, w.w1b), n)
        G(buf.R, _segments(x, w.wp1a), n)
    with TIMERS.span("gn_edge_gemms"):
        # edge_mlp layer 1 (+ReLU): h_e
        G(buf.he, _segments(e, w.w1c), ne, bias=hp(w.b1), relu=True,
          gather=[(buf.P.data.data_ptr(), ex.row_of.data_ptr()), (buf.Q.data.data_ptr(), idx.col.data_ptr())])
        # edge_mlp layer 2 (+ wrapper skip): the next layer's edge features
        e_next = None
        if need_edges_out:
            e_next = buf.e_alt
            G(e_next, _segments(buf.he, w.w2), ne, bias=hp(w.b2),
              residual=e.data.data_ptr() if skip else None, ldr=width)
        # phi layer 1 (+ReLU) on e1 = h_e W2^T + b2, folded
        G(buf.hm, _segments(buf.he, w.w3c), ne, bias=hp(w.b3c), relu=True,
          gather=[(buf.R.data.data_ptr(), idx.col.data_ptr())])
    # scatter_mean over row (phi layer 2 is folded into gamma layer 1)
    ws_bytes = capi.aggregate_workspace_bytes(idx.n_big)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.data.device)
    with TIMERS.span("gn_segment_mean"):
        capi.sage_aggregate(buf.hm.data.data_ptr(), buf.mh.data.data_ptr(), buf.hm.code, n, idx.rowptr.data_ptr(),
                            ex.iota.data_ptr(), idx.big_rows.data_ptr(), idx.n_big, capi.BG_AGGR_MEAN,
                            ws.data_ptr(), ws_bytes, _stream(), width=width)
    buf.mh.refresh_split()
    with TIMERS.span("gn_node_gemms"):
        gate_segs = _segments(ex.nonempty, w.wgate)[:2]      # the indicator is exact in tf32: its lo part is 0
        G(buf.g1, _segments(x, w.wg1a) + _segments(buf.mh, w.wgc) + gate_segs, n, bias=hp(w.bg1), relu=True)
        G(buf.xg, _segments(buf.g1, w.wg2), n, bias=hp(w.bg2))
        G(buf.t, _segments(buf.xg, w.wb1), n, bias=hp(w.bb1), relu=True)
        res = buf.xg
        if skip:                                   # x_next = xg + beta(xg) + x_prev
            add_into(buf.s, buf.xg, x)
            res = buf.s
        G(buf.x_alt, _segments(buf.t, w.wb2), n, bias=hp(w.bb2), residual=res.data.data_ptr(), ldr=width)
    x_next = buf.x_alt
    buf.x_alt = x                                  # ping-pong
    if e_next is not None:
        buf.e_alt = e
    return x_next, e_next


# ----------------------------------------------------------------------------- SAGPooling (GraphSAGE_SAG / EAGNN_SAG)
@dataclass
class SagPoolResult:
    """What PyG `SAGPooling.forward` returns (Models/BuckGNN.py:365-367, 502-504), plus the index maps."""
    x: Optional[Activation]       # [N', width] = x[perm] * score[perm]   (width 512, or 128: bg_*128)
    edge_index: torch.Tensor      # [2, E'] int64, relabelled, original edge order
    batch: torch.Tensor           # [N'] int64
    perm: torch.Tensor            # [N'] int32: old node id of each kept row
    score: torch.Tensor           # [N'] f32 = tanh score of the kept rows
    new_id: Optional[torch.Tensor]  # [N] int32: new row of an old node, -1 if dropped
    kept_edge: Optional[torch.Tensor]   # [E'] int32: old edge id of each kept edge
    n_nodes: int
    n_edges: int
    graph_ptr: torch.Tensor       # [G+1] int32 offsets of the pooled graphs
    all_scores: Optional[torch.Tensor]   # [N] f32 score of every node


def pool_summary(res: "SagPoolResult") -> "SagPoolResult":
    """The index side of a pooling result (what `self.pool` returns besides x): kept on the module for inspection
    without pinning the [N', 512] feature rows and the per-node scratch vectors in memory between calls."""
    import dataclasses
    return dataclasses.replace(res, x=None, new_id=None, all_scores=None)


def pack_sag_pool(pool) -> Dict[str, object]:
    gnn = pool.gnn
    f32 = lambda t: t.detach().float().contiguous().view(-1)
    return {"w_l": f32(gnn.lin_l.weight), "w_r": f32(gnn.lin_r.weight), "bias": float(gnn.lin_l.bias.detach().float().item()),
            "ratio": float(pool.ratio)}


def sag_pool(x: Activation, csr_by_target: GraphIndex, graph_ptr: torch.Tensor, n_graphs: int,
             edge_index: torch.Tensor, w: Dict[str, object], sign: float = 1.0, want_kept_edges: bool = False) -> SagPoolResult:
    """SAGPooling on the device: score GNN + per-graph top-k + row gather + edge filter.  Two result words
    (N', E') come back to the host through pinned memory -- PyG syncs at the same place (`num_nodes.max().item()`
    inside `topk`).  The row width of `x` picks the kernels: 512, or 128 (bg_sag_select128 / bg_gather_rows128)."""
    dev = x.data.device
    width = x.data.shape[1]
    select, gather = (capi.sag_select128, capi.gather_rows128) if width == 128 else (capi.sag_select, capi.gather_rows)
    n, g = csr_by_target.n_nodes, int(n_graphs)
    edge_index = edge_index.contiguous()
    e = edge_index.shape[1]
    s = _stream()
    f32 = dict(dtype=torch.float32, device=dev)
    i32 = dict(dtype=torch.int32, device=dev)
    score, score_sel = torch.empty(max(n, 1), **f32), torch.empty(max(n, 1), **f32)
    new_id, perm = torch.empty(max(n, 1), **i32), torch.empty(max(n, 1), **i32)
    batch_out = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    new_ptr = torch.empty(g + 1, **i32)
    info = torch.zeros(2, **i32)
    ws_bytes = capi.sag_workspace_bytes(n, e, g)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    idx = csr_by_target
    with TIMERS.span("sag_select"):
        select(x.data.data_ptr(), x.code, n, idx.rowptr.data_ptr(), idx.col.data_ptr(), idx.big_rows.data_ptr(),
               idx.n_big, w["w_l"].data_ptr(), w["w_r"].data_ptr(), w["bias"], float(sign),
               graph_ptr.data_ptr(), g, w["ratio"], edge_index.data_ptr(), e,
               score.data_ptr(), new_id.data_ptr(), perm.data_ptr(), batch_out.data_ptr(), score_sel.data_ptr(),
               new_ptr.data_ptr(), info.data_ptr(), ws.data_ptr(), ws_bytes, s)
    host = torch.zeros(2, dtype=torch.int32).pin_memory()
    capi.publish_words(info.data_ptr(), host.data_ptr(), 2, s)
    done = torch.cuda.Event()
    done.record()
    done.synchronize()
    n2, e2 = host.tolist()
    x_new = Activation(n2, width, x.precision, dev)
    ei_new = torch.empty((2, e2), dtype=torch.int64, device=dev)
    kept = torch.empty(max(e2, 1), **i32) if want_kept_edges else None
    with TIMERS.span("sag_connect"):
        gather(x.data.data_ptr(), x.code, width, perm.data_ptr(), score.data_ptr(), n2, x_new.data.data_ptr(), width, s)
        x_new.refresh_split()
        capi.sag_connect(edge_index.data_ptr(), e, n, new_id.data_ptr(), e2, ei_new.data_ptr(), _p(kept),
                         ws.data_ptr(), ws_bytes, s)
    return SagPoolResult(x_new, ei_new, batch_out[:n2], perm[:n2], score_sel[:n2], new_id[:n], kept, n2, e2, new_ptr,
                         score[:n])


def edge_slot_map(idx_old: GraphIndex, idx_new: GraphIndex, kept_edge: torch.Tensor) -> torch.Tensor:
    """[E'] int32: for every CSR slot of the pooled graph, the CSR slot of the same edge in the un-pooled graph."""
    dev = idx_old.rowptr.device
    s = _stream()
    e_old, e_new = idx_old.n_edges, idx_new.n_edges
    i32 = dict(dtype=torch.int32, device=dev)
    inv = torch.empty(max(e_old, 1), **i32)
    capi.index_invert(idx_old.perm.data_ptr(), e_old, inv.data_ptr(), s)            # old edge id -> old slot
    orig = torch.empty(max(e_new, 1), **i32)
    capi.index_gather(kept_edge.data_ptr(), idx_new.perm.data_ptr(), e_new, orig.data_ptr(), s)   # new slot -> old edge id
    slot = torch.empty(max(e_new, 1), **i32)
    capi.index_gather(inv.data_ptr(), orig.data_ptr(), e_new, slot.data_ptr(), s)   # new slot -> old slot
    return slot


def regather_edge_rows(e: Activation, idx_old: GraphIndex, idx_new: GraphIndex, kept_edge: torch.Tensor) -> Activation:
    """Edge features of the kept edges, moved from the old CSR slot order to the new one (EAGNN_SAG:
    `edge_attr[mask]` of PyG filter_adj, for edge tensors that live in CSR order), at the row width of `e`."""
    e_new = idx_new.n_edges
    width = e.data.shape[1]
    out = Activation(max(e_new, 1), width, e.precision, e.data.device)
    if e_new == 0:
        return out
    slot = edge_slot_map(idx_old, idx_new, kept_edge)
    gather = capi.gather_rows128 if width == 128 else capi.gather_rows
    gather(e.data.data_ptr(), e.code, width, slot.data_ptr(), None, e_new, out.data.data_ptr(), width, _stream())
    out.refresh_split()
    return out
