"""Training step of the EA-GNN ("CustomGNN") variants: `GraphNetBlock` (Models/BuckGNN.py:528-566) and its
wrapper loop (:326-336, :375-387) in train mode, forward and backward on the sm_100a kernels.

Forward of one block, as the reference writes it (edges live in CSR order keyed by `row = edge_index[0]`):
    he  = relu(cat[x[row], x[col], e] W1^T + b1)  = relu((x W1a^T)[row] + (x W1b^T)[col] + e W1c^T + b1)
    e1  = he W2^T + b2                                                       (the block's edge output)
    hm  = relu(cat[x[col], e1] Wp1^T + bp1)       = relu((x Wp1a^T)[col] + e1 Wp1b^T + bp1)
    m   = hm Wp2^T + bp2;   agg = scatter_mean(m, row)
    g1  = relu(cat[x, agg] Wg1^T + bg1);  xg = g1 Wg2^T + bg2
    t   = relu(xg Wb1^T + bb1);           xo = xg + t Wb2^T + bb2
    wrapper: x' = dropout(xo [+ x]),  e' = dropout(e1 [+ e])
Every product is `bg_gemm512` (gathered rows enter as epilogue addends); unlike the eval path nothing is
folded, so each Linear keeps its own input for its weight gradient.  Backward: the same kernel on transposed
weights for input gradients, `bg_wgrad512` for weight gradients (the reduction runs over nodes or edges),
`bg_grad_mask` for ReLU / Dropout, `bg_segment_expand` for scatter_mean, and `bg_sage_aggregate` over the two
CSR orders for the gathers' scatter-adds.

Width: EA_GNN / EA_GNN_Shared run at the model's hidden_channels, 512 or 128 (`BuckGNN.native128_eagnn_train`: a
hidden_channels = 128 model trains on its own 128-wide kernels instead of the zero-padded 512-wide twin of narrow.py).
At 128 the products run on `bg_gemm128` / `bg_gemm128_gathered` (engine.gemm picks by the output width), the weight
gradients on `bg_wgrad128_ld` (written in place into the column slices of the concatenated Linears, the pair
`[x | agg]` of node_mlp_gamma[0] in one launch), the row kernels are the `*128` entry points, and the encoders and the
decoder are the reference's 2-layer MLPs on bg_sgemm (train.py).  EAGNN_SAG trains at 512 only.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import capi, engine
from .engine import Activation, _stream
from .train import (GradStore, _Saved, _f32, colsum, encoder_backward, encoder_forward_train, head_backward,
                    head_forward_train, is_node_level, layer_seed, node_head_backward, node_head_forward_train,
                    split_k_layout, trainable_parameters, transposed_pack, weight_grad_mn)


def _blocks(model):
    if model.model_name == "EA_GNN_Shared":
        return [model.shared_gn_block] * model.num_layers
    return list(model.gn_blocks)


class _BlockWeights:
    """Operand-format slices of one GraphNetBlock (forward) and their transposes (backward), built on demand."""

    def __init__(self, blk, prec: str, width: int):
        self.blk, self.prec, self.W = blk, prec, width
        self._fwd, self._bwd = {}, {}

    def _slice(self, name):
        b, H = self.blk, self.W
        w1, wp1, wg1 = b.edge_mlp[0].weight, b.node_mlp_phi[0].weight, b.node_mlp_gamma[0].weight
        return {"w1a": w1[:, :H], "w1b": w1[:, H:2 * H], "w1c": w1[:, 2 * H:], "w2": b.edge_mlp[2].weight,
                "wp1a": wp1[:, :H], "wp1b": wp1[:, H:], "wp2": b.node_mlp_phi[2].weight,
                "wg1a": wg1[:, :H], "wg1b": wg1[:, H:], "wg2": b.node_mlp_gamma[2].weight,
                "wb1": b.node_mlp_beta[0].weight, "wb2": b.node_mlp_beta[2].weight}[name]

    def fwd(self, name):
        if name not in self._fwd:
            self._fwd[name] = engine.pack_linear(self._slice(name).detach().contiguous(), self.prec)
        return self._fwd[name]

    def bwd(self, name):
        if name not in self._bwd:
            self._bwd[name] = transposed_pack(self._slice(name).detach().contiguous(), self.prec)
        return self._bwd[name]


_BIAS_ORDER = ("b1", "b2", "bp1", "bp2", "bg1", "bg2", "bb1", "bb2")


def _bias_params(blk):
    return (blk.edge_mlp[0].bias, blk.edge_mlp[2].bias, blk.node_mlp_phi[0].bias, blk.node_mlp_phi[2].bias,
            blk.node_mlp_gamma[0].bias, blk.node_mlp_gamma[2].bias, blk.node_mlp_beta[0].bias, blk.node_mlp_beta[2].bias)


class _Stage:
    """One graph (n nodes, ne edges in CSR-by-row slot order) the GraphNetBlocks run on: the un-pooled batch, or the
    pooled one of EAGNN_SAG.  Holds the index structures and the small helpers of the forward / backward loops."""

    def __init__(self, idx, prec: str, dev, width: int, grads: Optional[GradStore] = None):
        self.idx, self.prec, self.dev, self.W = idx, prec, dev, width
        self.n, self.ne = idx.n_nodes, idx.n_edges
        self.code = engine.PRECISION_FORMATS[prec][0]
        self.ex = engine.edge_extras(idx, prec)
        self.grads = grads
        self._idx_c = None

    def mk(self, rows: int) -> Activation:
        return Activation(rows, self.W, self.prec, self.dev)

    def G(self, out, segs, m, **kw):
        engine.gemm(segs, m, self.prec, out, **kw)

    # ---- backward helpers
    @property
    def idx_c(self):
        """slots sorted by col: the scatter-add of a gradient that was gathered by `col` is a sum over this CSR"""
        if self._idx_c is None:
            ei_slots = torch.stack([self.ex.row_of[:self.ne].long(), self.idx.col[:self.ne].long()]).contiguous()
            self._idx_c = engine.build_graph_index(ei_slots, None, self.n, key_row=1)
        return self._idx_c

    def _sum_by(self, index, rowptr, big_rows, n_big, src: Activation) -> Activation:
        out = self.mk(self.n)
        nb = capi.aggregate_workspace_bytes(n_big)
        ws = torch.empty(nb, dtype=torch.uint8, device=self.dev)
        capi.sage_aggregate(src.data.data_ptr(), out.data.data_ptr(), self.code, self.n, rowptr.data_ptr(), index.data_ptr(),
                            big_rows.data_ptr(), n_big, capi.BG_AGGR_SUM, ws.data_ptr(), nb, _stream(), width=self.W)
        out.refresh_split()
        return out

    def by_row(self, src):
        return self._sum_by(self.ex.iota, self.idx.rowptr, self.idx.big_rows, self.idx.n_big, src)

    def by_col(self, src):
        c = self.idx_c
        return self._sum_by(c.perm, c.rowptr, c.big_rows, c.n_big, src)

    def masked(self, dy: Activation, act: Optional[Activation], rows: int, p: float = 0.0, sd: int = 0) -> Activation:
        out = self.mk(rows)
        capi.grad_mask(dy.data.data_ptr(), None, None if act is None else act.data.data_ptr(), out.data.data_ptr(), self.code,
                       rows, p, sd, _stream(), width=self.W)
        out.refresh_split()
        return out

    def linear_grads(self, dy: Activation, inp: Activation, rows: int, weight, col0: int, bias,
                     inp2: Optional[Activation] = None) -> None:
        """dW[:, col0:col0+W] += dy^T inp (and dW[:, col0+W:col0+2W] += dy^T inp2);  db += colsum(dy)  (bias None: a
        column slice that shares its bias)."""
        W = self.W
        with engine.TIMERS.span("train_wgrad"):
            dw = self.grads.zeros(weight)
            if W == 128:                                 # in place into the slices, inp2 in the same launch
                chunks, chunk_k = split_k_layout(rows, max_chunks=74)
                partial = _f32((chunks * 256, 128), self.dev)
                ld = dw.shape[1]
                with engine.TIMERS.span("train_wgrad_gemm"):
                    capi.wgrad128_ld(dy.data.data_ptr(), inp.data.data_ptr(), None if inp2 is None else inp2.data.data_ptr(),
                                     self.code, rows, chunks, chunk_k, partial.data_ptr(), dw[:, col0:].data_ptr(), ld,
                                     None if inp2 is None else dw[:, col0 + W:].data_ptr(), ld, True, _stream())
            else:
                for k, a in enumerate((inp, inp2)):
                    if a is None:
                        continue
                    tmp = _f32((W, W), self.dev)
                    weight_grad_mn(dy.data, a.data, self.code, rows, tmp, False)
                    dw[:, col0 + k * W:col0 + (k + 1) * W] += tmp
            if bias is not None:
                colsum(dy.data, self.code, rows, W, W, self.grads.zeros(bias), accumulate=True)

    def dgrad(self, dy: Activation, wt, rows: int, residual: Optional[Activation] = None) -> Activation:
        out = self.mk(rows)
        with engine.TIMERS.span("train_dgrad_gemm"):
            self.G(out, engine._segments(dy, wt), rows, residual=None if residual is None else residual.data.data_ptr(),
                   ldr=self.W)
        return out


def _block_forward(st: _Stage, blk, w: "_BlockWeights", bz, cur: Activation, e: Activation, skip: bool, p_drop: float,
                   seed: int, i: int, skip_after_dropout: bool):
    """One GraphNetBlock + the wrapper's skip / Dropout (Models/BuckGNN.py:378-386; `skip_after_dropout`: the order of
    the EAGNN_SAG loops, :356-373).  Returns (x_next, e_next, saved tuple)."""
    n, ne, idx, ex, code, W = st.n, st.ne, st.idx, st.ex, st.code, st.W
    s = _stream()
    seg, mk, G = engine._segments, st.mk, st.G
    hp = lambda t: t.data_ptr()
    row_of, col = ex.row_of.data_ptr(), idx.col.data_ptr()
    with engine.TIMERS.span("gn_node_gemms"):
        P, Q, R = mk(n), mk(n), mk(n)
        G(P, seg(cur, w.fwd("w1a")), n)
        G(Q, seg(cur, w.fwd("w1b")), n)
        G(R, seg(cur, w.fwd("wp1a")), n)
    with engine.TIMERS.span("gn_edge_gemms"):
        he, e1, hm, m = mk(ne), mk(ne), mk(ne), mk(ne)
        G(he, seg(e, w.fwd("w1c")), ne, bias=hp(bz["b1"]), relu=True, gather=[(P.data.data_ptr(), row_of), (Q.data.data_ptr(), col)])
        G(e1, seg(he, w.fwd("w2")), ne, bias=hp(bz["b2"]))
        G(hm, seg(e1, w.fwd("wp1b")), ne, bias=hp(bz["bp1"]), relu=True, gather=[(R.data.data_ptr(), col)])
        G(m, seg(hm, w.fwd("wp2")), ne, bias=hp(bz["bp2"]))
    agg = mk(n)
    agg_ws_bytes = capi.aggregate_workspace_bytes(idx.n_big)
    ws = torch.empty(agg_ws_bytes, dtype=torch.uint8, device=st.dev)
    with engine.TIMERS.span("gn_segment_mean"):
        capi.sage_aggregate(m.data.data_ptr(), agg.data.data_ptr(), code, n, idx.rowptr.data_ptr(), ex.iota.data_ptr(),
                            idx.big_rows.data_ptr(), idx.n_big, capi.BG_AGGR_MEAN, ws.data_ptr(), agg_ws_bytes, s, width=W)
    agg.refresh_split()
    del m, P, Q, R
    with engine.TIMERS.span("gn_node_gemms"):
        g1, xg, t, xo = mk(n), mk(n), mk(n), mk(n)
        G(g1, seg(cur, w.fwd("wg1a")) + seg(agg, w.fwd("wg1b")), n, bias=hp(bz["bg1"]), relu=True)
        G(xg, seg(g1, w.fwd("wg2")), n, bias=hp(bz["bg2"]))
        G(t, seg(xg, w.fwd("wb1")), n, bias=hp(bz["bb1"]), relu=True)
        G(xo, seg(t, w.fwd("wb2")), n, bias=hp(bz["bb2"]), residual=xg.data.data_ptr(), ldr=W)
    x_next, e_next = mk(n), mk(ne)
    inside = skip and not skip_after_dropout           # EA_GNN: dropout(x + x_prev);  EAGNN_SAG: dropout(x) + x_prev
    capi.dropout_residual(xo.data.data_ptr(), cur.data.data_ptr() if inside else None, x_next.data.data_ptr(), code, n,
                          p_drop, layer_seed(seed, 2 * i), s, width=W)
    capi.dropout_residual(e1.data.data_ptr(), e.data.data_ptr() if inside else None, e_next.data.data_ptr(), code, ne,
                          p_drop, layer_seed(seed, 2 * i + 1), s, width=W)
    if skip and skip_after_dropout:
        capi.add(x_next.data.data_ptr(), cur.data.data_ptr(), None, x_next.data.data_ptr(), code, x_next.data.numel(), s)
        capi.add(e_next.data.data_ptr(), e.data.data_ptr(), None, e_next.data.data_ptr(), code, e_next.data.numel(), s)
    x_next.refresh_split(); e_next.refresh_split()
    return x_next, e_next, (blk, cur, e, he, e1, hm, agg, g1, xg, t, skip)


def _block_backward(st: _Stage, saved, w: "_BlockWeights", dxn: Activation, den: Optional[Activation], p_drop: float,
                    seed: int, i: int, skip_after_dropout: bool):
    """Backward of `_block_forward`: (d x_next, d e_next or None) -> (d x_in, d e_in)."""
    n, ne, idx, code, W = st.n, st.ne, st.idx, st.code, st.W
    s = _stream()
    masked, linear_grads, dgrad, by_row, by_col, mk = st.masked, st.linear_grads, st.dgrad, st.by_row, st.by_col, st.mk
    blk, x_in, e_in, he, e1, hm, agg, g1, xg, t, skip = saved
    em, phi, gam, bet = blk.edge_mlp, blk.node_mlp_phi, blk.node_mlp_gamma, blk.node_mlp_beta
    dxo = masked(dxn, None, n, p_drop, layer_seed(seed, 2 * i))                   # Dropout backward
    de1 = None if den is None else masked(den, None, ne, p_drop, layer_seed(seed, 2 * i + 1))
    # what the skip branch receives: the dropped gradient when the skip sits inside the Dropout, the raw one otherwise
    skip_x = (dxn if skip_after_dropout else dxo) if skip else None
    skip_e = (den if skip_after_dropout else de1) if (skip and den is not None) else None
    # xo = xg + t Wb2^T + bb2;  t = relu(xg Wb1^T + bb1)
    linear_grads(dxo, t, n, bet[2].weight, 0, bet[2].bias)
    dt = masked(dgrad(dxo, w.bwd("wb2"), n), t, n)
    linear_grads(dt, xg, n, bet[0].weight, 0, bet[0].bias)
    dxg = dgrad(dt, w.bwd("wb1"), n, residual=dxo)
    # xg = g1 Wg2^T + bg2;  g1 = relu(cat[x, agg] Wg1^T + bg1)
    linear_grads(dxg, g1, n, gam[2].weight, 0, gam[2].bias)
    dg1 = masked(dgrad(dxg, w.bwd("wg2"), n), g1, n)
    linear_grads(dg1, x_in, n, gam[0].weight, 0, gam[0].bias, inp2=agg)            # [Wg1a | Wg1b]
    dx = dgrad(dg1, w.bwd("wg1a"), n, residual=skip_x)                             # + the wrapper's skip
    dagg = dgrad(dg1, w.bwd("wg1b"), n)
    # agg = scatter_mean(m, row);  m = hm Wp2^T + bp2;  hm = relu((x Wp1a^T)[col] + e1 Wp1b^T + bp1)
    dm = mk(ne)
    capi.segment_expand(dagg.data.data_ptr(), idx.rowptr.data_ptr(), n, True, dm.data.data_ptr(), code, s, width=W)
    dm.refresh_split()
    linear_grads(dm, hm, ne, phi[2].weight, 0, phi[2].bias)
    dhm = masked(dgrad(dm, w.bwd("wp2"), ne), hm, ne)
    del dm
    linear_grads(dhm, e1, ne, phi[0].weight, W, phi[0].bias)
    de1_tot = dgrad(dhm, w.bwd("wp1b"), ne, residual=de1)
    dR = by_col(dhm)
    del dhm
    linear_grads(dR, x_in, n, phi[0].weight, 0, None)
    dx = dgrad(dR, w.bwd("wp1a"), n, residual=dx)
    # e1 = he W2^T + b2;  he = relu((x W1a^T)[row] + (x W1b^T)[col] + e W1c^T + b1)
    linear_grads(de1_tot, he, ne, em[2].weight, 0, em[2].bias)
    dhe = masked(dgrad(de1_tot, w.bwd("w2"), ne), he, ne)
    linear_grads(dhe, e_in, ne, em[0].weight, 2 * W, em[0].bias)
    de_in = dgrad(dhe, w.bwd("w1c"), ne, residual=skip_e)
    dP, dQ = by_row(dhe), by_col(dhe)
    del dhe, de1_tot
    linear_grads(dP, x_in, n, em[0].weight, 0, None)
    linear_grads(dQ, x_in, n, em[0].weight, W, None)
    dx = dgrad(dP, w.bwd("w1a"), n, residual=dx)
    dx = dgrad(dQ, w.bwd("w1b"), n, residual=dx)
    return dx, de_in


def _block_tables(model, blocks, prec: str, width: int, extra_biases=()):
    """(biases tensor on the host, bias_of[id(block)], weights[id(block)], unique blocks): one read-back for every
    epilogue bias vector of the step."""
    uniq = []
    for b in blocks:
        if all(b is not q for q in uniq):
            uniq.append(b)
    bias_list = [model.node_encoder[-1].bias, model.edge_encoder[-1].bias] + list(extra_biases) + [p for b in uniq for p in _bias_params(b)]
    biases = torch.stack([b.detach().float() for b in bias_list]).cpu()
    off = 2 + len(extra_biases)
    bias_of = {id(b): {k: biases[off + 8 * j + i] for i, k in enumerate(_BIAS_ORDER)} for j, b in enumerate(uniq)}
    weights = {id(b): _BlockWeights(b, prec, width) for b in uniq}
    return biases, bias_of, weights


class EAGNNTrainFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, x, edge_index, edge_attr, batch, seed, *params):
        prec = model.train_precision
        dev = x.device
        x = x.detach().to(torch.float32).contiguous()
        if edge_attr is None or not edge_attr.is_cuda:
            raise RuntimeError("buckgnn_b200: `edge_attr` must be a CUDA tensor")
        n = x.shape[0]
        W = model.hidden_channels                          # 512, or 128 (BuckGNN.native128_eagnn_train)
        if W not in (512, 128):
            raise NotImplementedError(f"buckgnn_b200: the EA-GNN training step runs at width 512 or 128, not {W}")
        if W == 128 and is_node_level(model) and not model._runs_native128_node_head():
            raise NotImplementedError("buckgnn_b200: the 128-wide EA-GNN training step has node-level heads only with "
                                      "native128_node_head on")
        p_drop = float(model.dropout.p)
        pending = engine.begin_graph_index(edge_index, batch, n, key_row=0)       # GraphNetBlock aggregates on row (:553,561)
        blocks = _blocks(model)
        L = len(blocks)
        biases, bias_of, weights = _block_tables(model, blocks, prec, W)

        sv = _Saved()
        sv.model, sv.prec, sv.n, sv.x, sv.seed, sv.p_drop = model, prec, n, x, seed, p_drop
        sv.h1, sv.h2, cur = encoder_forward_train(model.node_encoder, x, prec, biases[0], width=W)       # :323
        idx = pending.finish()
        ne = idx.n_edges
        if ne == 0:
            raise NotImplementedError("buckgnn_b200: EA-GNN training needs at least one edge")
        sv.idx, sv.ne = idx, ne
        st = _Stage(idx, prec, dev, W)
        sv.stage = st
        # edge features in CSR order (input re-ordering only), then the edge encoder (:327, :376)
        ea = edge_attr.detach().to(torch.float32).index_select(0, idx.perm[:ne].long()).contiguous()
        sv.ea = ea
        sv.eh1, sv.eh2, e = encoder_forward_train(model.edge_encoder, ea, prec, biases[1], width=W)
        sv.layers = []
        for i, blk in enumerate(blocks):
            cur, e, saved = _block_forward(st, blk, weights[id(blk)], bias_of[id(blk)], cur, e, 0 < i < L - 1, p_drop, seed, i, False)
            sv.layers.append(saved)
        sv.weights = weights
        sv.node_level = is_node_level(model)
        pred = node_head_forward_train(model, cur, sv) if sv.node_level else head_forward_train(model, cur, idx, sv)
        ctx.sv = sv
        ctx.params = trainable_parameters(model)      # the module's own parameters key the GradStore (the inputs may be embeddings, narrow.py)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        sv = ctx.sv
        model, prec, n = sv.model, sv.prec, sv.n
        dev = sv.x.device
        grads = GradStore(dev, getattr(model, "_grad_sync", None))
        st = sv.stage
        st.grads = grads
        dxn = (node_head_backward if sv.node_level else head_backward)(
            model, sv, dpred.detach().to(torch.float32).contiguous(), n, prec, grads)
        den: Optional[Activation] = None                    # the last block's edge output feeds nothing
        for i in range(len(sv.layers) - 1, -1, -1):
            saved = sv.layers[i]
            dxn, den = _block_backward(st, saved, sv.weights[id(saved[0])], dxn, den, sv.p_drop, sv.seed, i, False)
        encoder_backward(model.node_encoder, sv.x, sv.h1, sv.h2, dxn, prec, grads)
        encoder_backward(model.edge_encoder, sv.ea, sv.eh1, sv.eh2, den, prec, grads)
        grads.finish()
        ctx.sv = None
        return (None, None, None, None, None, None, *grads.for_params(ctx.params))


class EAGNNSagTrainFunction(torch.autograd.Function):
    """Training step of `EAGNN_SAG` (Models/BuckGNN.py:219-244, 354-373): GraphNetBlocks, SAGPooling (node rows scaled by
    the tanh score, edge rows of the kept edges carried over), GraphNetBlocks on the pooled graph, pooling + head.  The
    skip is added after the Dropout in both loops (`i > 0` in the first, always in the second)."""

    @staticmethod
    def forward(ctx, model, x, edge_index, edge_attr, batch, seed, *params):
        prec = model.train_precision
        code = engine.PRECISION_FORMATS[prec][0]
        dev = x.device
        s = _stream()
        x = x.detach().to(torch.float32).contiguous()
        if edge_attr is None or not edge_attr.is_cuda:
            raise RuntimeError("buckgnn_b200: `edge_attr` must be a CUDA tensor")
        n = x.shape[0]
        p_drop = float(model.dropout.p)
        pending = engine.begin_graph_index(edge_index, batch, n, key_row=0)       # GraphNetBlock direction (source-keyed)
        pending_t = engine.begin_graph_index(edge_index, None, n, key_row=1)      # SAGEConv direction of the score GNN
        first, second = list(model.gnn_layers_1), list(model.gnn_layers_2)
        W = 512                                            # EAGNN_SAG trains at 512 (the twin at other widths)
        biases, bias_of, weights = _block_tables(model, first + second, prec, W)
        sv = _Saved()
        sv.model, sv.prec, sv.n, sv.x, sv.seed, sv.p_drop = model, prec, n, x, seed, p_drop
        sv.h1, sv.h2, cur = encoder_forward_train(model.node_encoder, x, prec, biases[0])
        idx = pending.finish()
        idx_t = pending_t.finish()
        ne = idx.n_edges
        if ne == 0:
            raise NotImplementedError("buckgnn_b200: EA-GNN training needs at least one edge")
        st1 = _Stage(idx, prec, dev, W)
        ea = edge_attr.detach().to(torch.float32).index_select(0, idx.perm[:ne].long()).contiguous()
        sv.ea = ea
        sv.eh1, sv.eh2, e = encoder_forward_train(model.edge_encoder, ea, prec, biases[1])
        sv.first, sv.second = [], []
        for i, blk in enumerate(first):
            cur, e, saved = _block_forward(st1, blk, weights[id(blk)], bias_of[id(blk)], cur, e, i > 0, p_drop, seed, i, True)
            sv.first.append(saved)
        # ---- SAGPooling (:365-367)
        pack = engine.pack_sag_pool(model.pool)
        pooled = engine.sag_pool(cur, idx_t, idx.graph_ptr, idx.n_graphs, edge_index, pack, sign=model._sag_sign, want_kept_edges=True)
        model.last_pool = engine.pool_summary(pooled)   # perm / score / edge_index / batch of the last pooling, without its feature rows
        idx2 = engine.build_graph_index(pooled.edge_index, pooled.batch, pooled.n_nodes, key_row=0)
        if idx2.n_edges == 0:
            raise NotImplementedError("buckgnn_b200: EAGNN_SAG training needs at least one edge after the pooling")
        slot_map = engine.edge_slot_map(idx, idx2, pooled.kept_edge)             # new slot -> old slot
        e2 = Activation(idx2.n_edges, W, prec, dev)
        capi.gather_rows(e.data.data_ptr(), code, W, slot_map.data_ptr(), None, idx2.n_edges, e2.data.data_ptr(), W, s)
        e2.refresh_split()
        sv.pool_in, sv.pooled, sv.pool_pack, sv.slot_map = cur, pooled, pack, slot_map
        st2 = _Stage(idx2, prec, dev, W)
        cur, e = pooled.x, e2
        k0 = len(first)
        for k, blk in enumerate(second):
            cur, e, saved = _block_forward(st2, blk, weights[id(blk)], bias_of[id(blk)], cur, e, True, p_drop, seed, k0 + k, True)
            sv.second.append(saved)
        sv.st1, sv.st2, sv.weights = st1, st2, weights
        sv.idx = idx2                                   # head_backward reads sv.idx.graph_ptr
        pred = head_forward_train(model, cur, idx2, sv)
        ctx.sv = sv
        ctx.params = trainable_parameters(model)      # the module's own parameters key the GradStore (the inputs may be embeddings, narrow.py)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        sv = ctx.sv
        model, prec, n = sv.model, sv.prec, sv.n
        dev = sv.x.device
        s = _stream()
        F32 = capi.BG_F32
        grads = GradStore(dev, getattr(model, "_grad_sync", None))
        st1, st2 = sv.st1, sv.st2
        st1.grads = st2.grads = grads
        code = st1.code
        pooled = sv.pooled
        n2 = pooled.n_nodes
        dxn = head_backward(model, sv, dpred.detach().to(torch.float32).contiguous(), n2, prec, grads)
        den: Optional[Activation] = None
        k0 = len(sv.first)
        for k in range(len(sv.second) - 1, -1, -1):
            saved = sv.second[k]
            dxn, den = _block_backward(st2, saved, sv.weights[id(saved[0])], dxn, den, sv.p_drop, sv.seed, k0 + k, True)
        # ---- SAGPooling backward: node rows through x[perm] * tanh(score) and the scorer, edge rows back to their slots
        idx = st1.idx                                    # keyed by source: the transposed 'add' aggregation of the scorer
        xin = sv.pool_in
        W = st1.W
        dx = Activation(n, W, prec, dev)
        t, dpre = _f32((n,), dev), _f32((n,), dev)
        pack = sv.pool_pack
        with engine.TIMERS.span("sag_pool_bwd"):
            capi.sag_pool_backward(dxn.data.data_ptr(), xin.data.data_ptr(), code, n, n2, pooled.perm.data_ptr(),
                                   pooled.new_id.data_ptr(), pooled.all_scores.data_ptr(), float(model._sag_sign),
                                   idx.rowptr.data_ptr(), idx.col.data_ptr(), idx.big_rows.data_ptr(), idx.n_big,
                                   pack["w_l"].data_ptr(), pack["w_r"].data_ptr(), dx.data.data_ptr(), t.data_ptr(),
                                   dpre.data_ptr(), s)
            dx.refresh_split()
            gnn = model.pool.gnn
            dwl, _ = grads.get(gnn.lin_l.weight); dwr, _ = grads.get(gnn.lin_r.weight); dbl, _ = grads.get(gnn.lin_l.bias)
            from .train import sgemm
            sgemm(t, F32, 0, 1, xin.data, code, W, 1, 1, W, n, dwl, F32, W)
            sgemm(dpre, F32, 0, 1, xin.data, code, W, 1, 1, W, n, dwr, F32, W)
            colsum(dpre, F32, n, 1, 1, dbl)
            de = None
            if den is not None:
                ne, ne2 = st1.ne, st2.ne
                inv = torch.full((ne,), -1, dtype=torch.int32, device=dev)     # old slot -> new slot, -1 for a dropped edge
                capi.index_invert(sv.slot_map.data_ptr(), ne2, inv.data_ptr(), s)
                de = Activation(ne, W, prec, dev)
                capi.gather_rows(den.data.data_ptr(), code, W, inv.data_ptr(), None, ne, de.data.data_ptr(), W, s)
                de.refresh_split()
        dxn, den = dx, de
        for i in range(len(sv.first) - 1, -1, -1):
            saved = sv.first[i]
            dxn, den = _block_backward(st1, saved, sv.weights[id(saved[0])], dxn, den, sv.p_drop, sv.seed, i, True)
        encoder_backward(model.node_encoder, sv.x, sv.h1, sv.h2, dxn, prec, grads)
        if den is not None:
            encoder_backward(model.edge_encoder, sv.ea, sv.eh1, sv.eh2, den, prec, grads)
        grads.finish()
        ctx.sv = None
        return (None, None, None, None, None, None, *grads.for_params(ctx.params))
