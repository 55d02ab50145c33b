"""hidden_channels != 512 on the 512-wide kernels, by exact zero padding.

The reference's shipped configurations use `hidden_channels=128` (`TRAIN_FINAL.py:55,71`, the constructor default
`Models/BuckGNN.py:10`); the thesis model is 512 wide (`README.md:53-57`).  The eval forward of a 128-wide GraphSAGE
model with a graph-level head runs on its own 128-wide kernels (`BuckGNN._forward_cuda(width=128)`, bg_gemm128), and so
does that of EA_GNN / EA_GNN_Shared when `native128_eagnn` is on (`BuckGNN._forward_cuda_eagnn(width=128)`,
bg_gemm128_gathered).  Node-level heads of those models run 128 wide, in eval and training, when `native128_node_head`
is on (bg_node_head128 in eval), and so do GraphSAGE_SAG / EAGNN_SAG when `native128_sag` is on (eval with every head,
training with the eigenvalue head; bg_sag_select128).  What has no narrow kernels -- EA-GNN by default, the SAGPooling
variants and node-level heads without their flags, widths 64 / 256 -- and training without `native128_train`
(EA_GNN / EA_GNN_Shared: `native128_eagnn_train`) runs as the model's zero-padded 512-wide twin:

* every `[h, h]` weight sits in the top-left corner of a `[512, 512]` one, biases / BatchNorm affine terms are padded
  with zeros (running_var with ones): padded activation columns are exactly 0 through Linear, L2-normalize (the norm
  over 512 columns equals the norm over h), BatchNorm, ReLU, skip and dropout, so the first h columns are exactly the
  narrow model's;
* `cat[a, b, c] W^T` weights (`GraphNetBlock`, `Models/BuckGNN.py:531-545`; the `supernode_with_pooling` decoder,
  `:55-58, 85-92`) are padded per h-wide column block;
* h <= 128 has two-layer encoders / decoder (`Models/BuckGNN.py:41-65`): `Linear(F, 64), ReLU, Linear(64, h)` runs as
  `Linear(F, 64), ReLU, Linear(64, 128) = [I; 0], ReLU, Linear(128, 512) = pad(W)` -- the inserted ReLU acts on values
  that are already >= 0 -- and `Linear(h, 64), ReLU, Linear(64, out)` as `Linear(512, 128) = [pad(W); 0], ReLU,
  Linear(128, 64) = [I, 0], ReLU, Linear(64, out)`.

The embedding is a differentiable re-layout of the parameters (torch pad / cat: weight plumbing, no activation math),
so in train mode autograd slices the twin's gradients back onto the narrow parameters; BatchNorm running statistics are
copied back after a train-mode forward.  16x (h = 128) / 4x (h = 256) of the tensor work multiplies zeros: this path is
for compatibility with the shipped scripts, the measured configuration is h = 512.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

WIDE = 512


def _pad2(w: torch.Tensor, rows: int, cols: int) -> torch.Tensor:
    return F.pad(w, (0, cols - w.shape[1], 0, rows - w.shape[0]))


def _pad1(b: torch.Tensor, n: int, value: float = 0.0) -> torch.Tensor:
    return F.pad(b, (0, n - b.shape[0]), value=value)


def _pad_blocks(w: torch.Tensor, h: int, rows: int) -> torch.Tensor:
    """[r, k*h] -> [rows, k*512]: every h-wide column block padded to 512 columns."""
    k = w.shape[1] // h
    return torch.cat([_pad2(w[:, i * h:(i + 1) * h], rows, WIDE) for i in range(k)], dim=1)


class WideTwin:
    """The 512-wide twin of a narrow `BuckGNN` and the parameter / buffer embeddings between the two."""

    def __init__(self, narrow, ctor_kwargs: Dict[str, object]):
        from .model import BuckGNN
        self.narrow = narrow
        kw = dict(ctor_kwargs)
        kw["hidden_channels"] = WIDE
        self.twin = BuckGNN(**kw)
        self.h = h = narrow.hidden_channels
        self.params: List[Tuple[nn.Parameter, Callable[[], torch.Tensor]]] = []   # twin parameter <- embedding of narrow ones
        self.consts: List[Tuple[nn.Parameter, torch.Tensor]] = []
        self.bn_pairs: List[Tuple[nn.BatchNorm1d, nn.BatchNorm1d]] = []           # (twin BatchNorm, narrow BatchNorm)
        n, t = narrow, self.twin
        two_layer = h <= 128
        for enc_n, enc_t in ((n.node_encoder, t.node_encoder), (n.edge_encoder, t.edge_encoder)):
            self._same(enc_t[0], enc_n[0])
            if two_layer:
                eye = torch.zeros(128, 64)
                eye[:64] = torch.eye(64)
                self._const(enc_t[2].weight, eye)
                self._const(enc_t[2].bias, torch.zeros(128))
                self._lin(enc_t[4], enc_n[2], WIDE, 128)
            else:
                self._same(enc_t[2], enc_n[2])
                self._lin(enc_t[4], enc_n[4], WIDE, 128)
        dn, dt = n.decoder, t.decoder
        if two_layer:
            self._add(dt[0].weight, lambda w=dn[0].weight: _pad_blocks(w, h, 128))
            self._add(dt[0].bias, lambda b=dn[0].bias: _pad1(b, 128))
            eye = torch.zeros(64, 128)
            eye[:, :64] = torch.eye(64)
            self._const(dt[2].weight, eye)
            self._const(dt[2].bias, torch.zeros(64))
            self._same(dt[4], dn[2])
        else:
            self._add(dt[0].weight, lambda w=dn[0].weight: _pad_blocks(w, h, 128))
            self._add(dt[0].bias, lambda b=dn[0].bias: b)
            self._same(dt[2], dn[2])
            self._same(dt[4], dn[4])
        self._lin(t.pooling_mpl.mlp[0], n.pooling_mpl.mlp[0], WIDE, WIDE)
        for name in ("shared_gn_block",):
            if hasattr(n, name):
                self._gnblock(getattr(t, name), getattr(n, name))
        for name in ("gn_blocks", "gnn_layers_1", "gnn_layers_2"):
            if hasattr(n, name):
                for bt, bn_ in zip(getattr(t, name), getattr(n, name)):
                    self._gnblock(bt, bn_)
        if hasattr(n, "shared_graphsage_block"):
            self._sage(t.shared_graphsage_block, n.shared_graphsage_block)
        for name in ("sage_blocks_sum", "sage_blocks_add", "sage_blocks_mean", "sage_blocks_max", "sage_layers_1", "sage_layers_2"):
            if hasattr(n, name):
                for ct, cn in zip(getattr(t, name), getattr(n, name)):
                    self._sage(ct, cn)
        for name in ("batch_norms", "batch_norms_1", "batch_norms_2"):
            if hasattr(n, name):
                for bt, bn_ in zip(getattr(t, name), getattr(n, name)):
                    self._bn(bt, bn_)
        if hasattr(n, "pool"):
            g_t, g_n = t.pool.gnn, n.pool.gnn
            self._add(g_t.lin_l.weight, lambda w=g_n.lin_l.weight: _pad2(w, 1, WIDE))
            self._add(g_t.lin_l.bias, lambda b=g_n.lin_l.bias: b)
            self._add(g_t.lin_r.weight, lambda w=g_n.lin_r.weight: _pad2(w, 1, WIDE))
        for p in self.twin.parameters():
            p.requires_grad_(False)              # the twin holds values; gradients flow through the embeddings

    # ---- mapping builders
    def _add(self, twin_param, fn):
        self.params.append((twin_param, fn))

    def _const(self, twin_param, value):
        self.consts.append((twin_param, value))

    def _same(self, lin_t, lin_n):
        self._add(lin_t.weight, lambda w=lin_n.weight: w)
        self._add(lin_t.bias, lambda b=lin_n.bias: b)

    def _lin(self, lin_t, lin_n, rows, cols):
        self._add(lin_t.weight, lambda w=lin_n.weight: _pad2(w, rows, cols))
        if lin_n.bias is not None:
            self._add(lin_t.bias, lambda b=lin_n.bias: _pad1(b, rows))

    def _sage(self, ct, cn):
        self._lin(ct.lin_l, cn.lin_l, WIDE, WIDE)
        self._add(ct.lin_r.weight, lambda w=cn.lin_r.weight: _pad2(w, WIDE, WIDE))

    def _gnblock(self, bt, bn_):
        h = self.h
        for seq in ("edge_mlp", "node_mlp_phi", "node_mlp_gamma", "node_mlp_beta"):
            st, sn = getattr(bt, seq), getattr(bn_, seq)
            self._add(st[0].weight, lambda w=sn[0].weight: _pad_blocks(w, h, WIDE))
            self._add(st[0].bias, lambda b=sn[0].bias: _pad1(b, WIDE))
            self._lin(st[2], sn[2], WIDE, WIDE)

    def _bn(self, bt, bn_):
        self._add(bt.weight, lambda w=bn_.weight: _pad1(w, WIDE))
        self._add(bt.bias, lambda b=bn_.bias: _pad1(b, WIDE))
        self.bn_pairs.append((bt, bn_))       # buffers are looked up at use time: Module.to() replaces buffer tensors

    # ---- use
    def _signature(self):
        n = self.narrow
        return tuple((p.data_ptr(), p._version) for p in n.parameters()) + tuple((b.data_ptr(), b._version) for b in n.buffers())

    def sync(self, differentiable: bool) -> Dict[int, torch.Tensor]:
        """Refreshes the twin's parameter / buffer values from the narrow model.  With `differentiable`, returns
        {id(twin parameter): embedded tensor connected to the narrow parameters by autograd}."""
        dev = next(self.narrow.parameters()).device
        if next(self.twin.parameters()).device != dev:
            self.twin.to(dev)
        self.twin.train(self.narrow.training)
        self.twin.dropout.p = self.narrow.dropout.p
        sig = self._signature()
        if not differentiable and getattr(self, "_sig", None) == sig:
            return {}
        live: Dict[int, torch.Tensor] = {}
        with torch.set_grad_enabled(differentiable):
            vals = [fn() for _, fn in self.params]
        with torch.no_grad():
            for (tp, _), v in zip(self.params, vals):
                tp.copy_(v)                      # in place on the twin's leaf: bumps its version -> operand packs rebuild
                if differentiable and v.requires_grad:
                    live[id(tp)] = v
            for tp, value in self.consts:
                tp.copy_(value.to(dev))
            for bt, bn_ in self.bn_pairs:
                h = bn_.num_features
                bt.running_mean.zero_()
                bt.running_mean[:h].copy_(bn_.running_mean)
                bt.running_var.fill_(1.0)
                bt.running_var[:h].copy_(bn_.running_var)
                bt.num_batches_tracked.copy_(bn_.num_batches_tracked)
                bt.momentum, bt.eps = bn_.momentum, bn_.eps
        self._sig = None if differentiable else sig
        return live

    def copy_back_buffers(self) -> None:
        """BatchNorm running statistics written by a train-mode forward of the twin -> the narrow model's buffers."""
        with torch.no_grad():
            for bt, bn_ in self.bn_pairs:
                h = bn_.num_features
                bn_.running_mean.copy_(bt.running_mean[:h])
                bn_.running_var.copy_(bt.running_var[:h])
                bn_.num_batches_tracked.copy_(bt.num_batches_tracked)

    def forward(self, x, edge_index, edge_attr, batch):
        n, t = self.narrow, self.twin
        if not n.training:
            self.sync(differentiable=False)
            out = t(x, edge_index, edge_attr, batch)
        else:
            live = self.sync(differentiable=torch.is_grad_enabled())
            t._param_inputs = live
            try:
                out = t(x, edge_index, edge_attr, batch)
            finally:
                t._param_inputs = None
            self.copy_back_buffers()
        if hasattr(t, "last_pool"):
            n.last_pool = t.last_pool
        return out
