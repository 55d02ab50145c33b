"""Training step of the GraphSAGE BuckGNN on the sm_100a kernels (BASELINE.json configs[3]).

`TRAIN_FINAL.py:289-297` of the reference does `model.train(); pred, _ = model(...); loss.backward();
optimizer.step()`.  In train mode `BuckGNN.forward` routes here: one `torch.autograd.Function` whose
forward and backward are sequences of C-ABI calls (include/buckgnn_b200.h, "training step"); torch
provides memory, streams and the autograd graph edge between `pred` and the parameters, nothing else.

Per layer (Models/BuckGNN.py:447-458, train mode)
    forward   agg = A x                                   bg_sage_aggregate            (saved)
              u = normalize(agg Wl^T + b + x Wr^T)        bg_gemm512, inv_norm_out     (saved, with 1/|z|)
              batch statistics of u -> a, shift           bg_bn_batch_stats (+ running stats, momentum)
              y = dropout(relu(a u + shift) + x_prev)     bg_bn_act_forward (counter-based mask)
    backward  dz, dgamma, dbeta                           bg_sage_backward_rows
              dWl = dz^T agg, dWr = dz^T x                bg_wgrad512 (MN-major operands, split over nodes) + bg_reduce_partials
              db = colsum(dz)                             bg_colsum
              dagg = (dz / deg) Wl                        bg_gemm512 on the transposed weight
              dx = dz Wr + A^T dagg  (+ g on skip layers) bg_sage_aggregate over the CSR keyed by source + bg_gemm512
The encoder's first two Linears, the decoder and their gradients run on `bg_sgemm` (fp32 CUDA cores).

Width: the step runs at the model's hidden_channels, 512 or 128 (`BuckGNN.native128_train`: a hidden_channels = 128
model trains on its own 128-wide kernels -- bg_gemm128, bg_wgrad128 and the `*128` row kernels -- instead of the
zero-padded 512-wide twin of narrow.py).  At 128 the encoder and decoder are the reference's 2-layer MLPs
(Models/BuckGNN.py:41-65), all on bg_sgemm.  Node-level heads train at 128 when `BuckGNN.native128_node_head` is on.

Precision: `train_precision` in {"tf32" (default; fp32 storage), "bf16", "fp16"}: activations, saved tensors and
gradients of activations are stored in that format, weight gradients and all reductions are fp32.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import capi, engine
from .engine import Activation, _p, _stream

_GOLDEN = 0x9E3779B97F4A7C15
_MASK64 = (1 << 64) - 1


def layer_seed(seed: int, layer: int) -> int:
    return (seed + (layer + 1) * _GOLDEN) & _MASK64


def _f32(shape, dev):
    return torch.empty(shape, dtype=torch.float32, device=dev)


def _ws(nbytes, dev):
    return torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)


def sgemm(a, a_code, sam, sak, b, b_code, sbk, sbn, m, n, k, out, out_code, ldo, *, bias=None, relu=False,
          mask=None, mask_code=capi.BG_F32, mask_ld=0, accumulate=False):
    """out[m,n] (+)= mask(relu(sum_k a[m*sam + k*sak] * b[k*sbk + n*sbn] + bias[n]))   (bg_sgemm)."""
    nbytes = capi.sgemm_workspace_bytes(m, n, k)
    ws = _ws(nbytes, out.device)
    capi.sgemm(a.data_ptr(), a_code, sam, sak, b.data_ptr(), b_code, sbk, sbn, m, n, k, _p(bias), relu,
               _p(mask), mask_code, mask_ld, out.data_ptr(), out_code, ldo, accumulate, ws.data_ptr(), nbytes, _stream())


def colsum(src, code, rows, cols, ld, out, accumulate=False):
    nbytes = capi.colsum_workspace_bytes(rows, cols)
    ws = _ws(nbytes, out.device)
    capi.colsum(src.data_ptr(), code, rows, cols, ld, out.data_ptr(), accumulate, ws.data_ptr(), nbytes, _stream())


def split_k_layout(n_rows: int, max_chunks: int = 37):
    """(chunks, chunk_k) of the split over nodes for the weight-gradient GEMMs: one 512 x 512 product (width 128:
    max_chunks = 74, one 256 x 128 tile) per CTA pair of the 148-SM part when there is enough work, K per chunk a
    multiple of 64."""
    chunks = max(1, min(max_chunks, -(-n_rows // 1024)))
    chunk_k = -(-(-(-n_rows // chunks)) // 64) * 64
    return chunks, chunk_k


class ChunkedTranspose:
    """[N, C] activation -> [chunks][C][chunk_k] (bg_transpose_chunks): node dimension contiguous."""

    def __init__(self, act: torch.Tensor, code: int, n_rows: int, chunks: int, chunk_k: int, pad_rows: int = 0):
        """pad_rows > cols: every chunk is padded with zero rows to `pad_rows` (a narrow matrix made the
        512-row B operand of the split-K GEMM)."""
        cols = act.shape[1]
        rows = max(cols, pad_rows)
        alloc = torch.zeros if rows > cols else torch.empty
        self.data = alloc((chunks * rows, chunk_k), dtype=act.dtype, device=act.device)
        self.code, self.chunks, self.chunk_k, self.cols = code, chunks, chunk_k, cols
        capi.transpose_chunks(act.data_ptr(), code, n_rows, cols, act.shape[1], chunks, chunk_k,
                              self.data.data_ptr(), _stream(), out_rows_per_chunk=rows)


def weight_grad_512(dz_t: ChunkedTranspose, act_t: ChunkedTranspose, precision: str, out: torch.Tensor,
                    accumulate: bool) -> None:
    """out[o, i] (+)= sum_n dz[n, o] act[n, i]  -- `chunks` independent 512x512xchunk_k products on tcgen05
    (fp32 partials), then a fixed-order sum over the chunks."""
    s, kc = dz_t.chunks, dz_t.chunk_k
    dev = out.device
    partial = _f32((s * 512, 512), dev)
    a_code, b_code = engine.PRECISION_FORMATS[precision]
    with engine.TIMERS.span("train_wgrad_gemm"):
        capi.gemm512([(dz_t.data.data_ptr(), kc, act_t.data.data_ptr(), kc, kc)], s * 512, a_code, b_code,
                     partial.data_ptr(), capi.BG_F32, 512, _stream(), b_groups=s)
    capi.reduce_partials(partial.data_ptr(), s, 512 * 512, out.data_ptr(), accumulate, _stream())


def weight_grad_mn(dz: torch.Tensor, act: torch.Tensor, code: int, n_rows: int, out: torch.Tensor, accumulate: bool) -> None:
    """out[o, i] (+)= sum_n dz[n, o] act[n, i], dz [n, 512] and act [n, <= 512] read in place as MN-major tcgen05
    operands (bg_wgrad512): no transposed copies.  `out` is [512, 512] f32."""
    chunks, chunk_k = split_k_layout(n_rows)
    partial = _f32((chunks * 512, 512), out.device)
    with engine.TIMERS.span("train_wgrad_gemm"):
        capi.wgrad512(dz.data_ptr(), dz.shape[1], act.data_ptr(), act.shape[1], act.shape[1], code, n_rows, chunks,
                      chunk_k, partial.data_ptr(), _stream())
    capi.reduce_partials(partial.data_ptr(), chunks, 512 * 512, out.data_ptr(), accumulate, _stream())


def sage_weight_grads(dz: torch.Tensor, agg: torch.Tensor, x: torch.Tensor, code: int, n_rows: int, dwl: torch.Tensor,
                      acc_l: bool, dwr: torch.Tensor, acc_r: bool) -> None:
    """dWl (+)= dz^T agg and dWr (+)= dz^T x of one SAGE layer at the rows' width: two bg_wgrad512 products at 512,
    one bg_wgrad128 launch for both at 128."""
    width = dz.shape[1]
    if width == 512:
        weight_grad_mn(dz, agg, code, n_rows, dwl, acc_l)
        weight_grad_mn(dz, x, code, n_rows, dwr, acc_r)
        return
    if acc_l != acc_r:
        raise RuntimeError("buckgnn_b200: lin_l and lin_r of a layer accumulate together")
    chunks, chunk_k = split_k_layout(n_rows, max_chunks=74)
    partial = _f32((chunks * 256, 128), dz.device)
    with engine.TIMERS.span("train_wgrad_gemm"):
        capi.wgrad128(dz.data_ptr(), agg.data_ptr(), x.data_ptr(), code, n_rows, chunks, chunk_k, partial.data_ptr(),
                      dwl.data_ptr(), dwr.data_ptr(), acc_l, _stream())


def transposed_pack(weight: torch.Tensor, precision: str) -> engine.LinearPack:
    """W^T in operand format: the B operand of dX = dZ W (rows = input features)."""
    w = weight.detach().to(torch.float32).contiguous()
    wt = torch.empty((w.shape[1], w.shape[0]), dtype=torch.float32, device=w.device)
    capi.transpose_chunks(w.data_ptr(), capi.BG_F32, w.shape[0], w.shape[1], w.shape[1], 1, w.shape[0],
                          wt.data_ptr(), _stream())
    return engine.pack_linear(wt, precision)


class _Saved:
    pass


class GradStore:
    """fp32 gradient buffers by parameter; the second touch of a parameter (shared blocks) accumulates."""

    def __init__(self, device, sync=None):
        """`sync` (dist.GradSync): gradients are written into slices of its flat all-reduce buffer and handed to the
        collective group by group (`done`), overlapping the rest of the backward."""
        self.device, self.bufs, self.sync = device, {}, sync
        if sync is not None:
            sync.begin_step()

    def _new(self, param):
        if self.sync is not None:
            v = self.sync.view(param)
            if v is not None:
                return v
        return _f32(tuple(param.shape), self.device)

    def get(self, param):
        """(buffer, accumulate?) -- the caller overwrites a fresh buffer completely."""
        t = self.bufs.get(id(param))
        fresh = t is None
        if fresh:
            t = self.bufs[id(param)] = self._new(param)
        return t, not fresh

    def zeros(self, param):
        """A zero-initialised buffer that column slices are ADDED into."""
        t = self.bufs.get(id(param))
        if t is None:
            t = self.bufs[id(param)] = self._new(param)
            t.zero_()
        return t

    def done(self, params) -> None:
        """The gradients of `params` are final (no later layer of the backward adds to them)."""
        if self.sync is not None:
            self.sync.launch([p_ for p_ in params if p_ is not None and id(p_) in self.bufs])

    def finish(self) -> None:
        if self.sync is not None:
            self.sync.finish()

    def for_params(self, params):
        out: List[Optional[torch.Tensor]] = []
        snap = None
        if self.sync is not None:
            # autograd may adopt a returned gradient as `.grad` without copying; the flat all-reduce buffer is reused by
            # the next step, so hand out slices of a per-step snapshot instead (one copy kernel for all parameters)
            snap = self.sync.flat.clone()
        for p_ in params:
            t = self.bufs.get(id(p_))
            if t is not None and snap is not None and self.sync.view(p_) is not None:
                off, n, shape = self.sync.offsets[id(p_)]
                t = snap[off:off + n].view(shape)
            out.append(None if t is None else t.to(p_.dtype))
        return out


# ----------------------------------------------------------------------------- shared pieces: encoders and head
def _mat(t):
    """(tensor, format code) of an fp32 matrix or of an Activation in its storage format."""
    return (t.data, t.code) if isinstance(t, Activation) else (t, capi.BG_F32)


def _linears(seq):
    """[(nn.Linear, whether an nn.ReLU follows it)] of an nn.Sequential."""
    mods = list(seq)
    return [(m, isinstance(nxt, torch.nn.ReLU)) for m, nxt in zip(mods, mods[1:] + [None])
            if isinstance(m, torch.nn.Linear)]


def chain_forward(chain, x, out: Optional[Activation] = None):
    """y = L_k(..relu(L_1(x))..) for chain = [(nn.Linear, relu after)], one bg_sgemm per Linear.  `x` is fp32 or an
    Activation; every intermediate is fp32, and so is y unless `out` (an Activation) is given.  Returns (y, the input
    of every Linear): the operands of `chain_backward`."""
    F32 = capi.BG_F32
    m = _mat(x)[0].shape[0]
    xs = []
    for i, (lin, relu) in enumerate(chain):
        w, b = lin.weight.detach().float().contiguous(), lin.bias.detach().float().contiguous()
        n_out, k = w.shape
        y = out if out is not None and i == len(chain) - 1 else _f32((m, n_out), w.device)
        (xd, xc), (yd, yc) = _mat(x), _mat(y)
        sgemm(xd, xc, k, 1, w, F32, 1, k, m, n_out, k, yd, yc, n_out, bias=b, relu=relu)
        xs.append(x)
        x = y
    if out is not None:
        out.refresh_split()
    return x, xs


def chain_backward(chain, xs, dy, grads: GradStore, dx=None):
    """Backward of `chain_forward` given dy = d(y) (fp32 or an Activation), last Linear first: dW = dy^T x,
    db = colsum(dy), then d(x) = dy W, masked by x > 0 where x is the output of a ReLU of the chain.  The gradient of
    the chain's input goes to `dx` (fp32 or an Activation) and is not computed without one; the others are fp32."""
    F32 = capi.BG_F32
    m = _mat(xs[0])[0].shape[0]
    for i in range(len(chain) - 1, -1, -1):
        lin = chain[i][0]
        w = lin.weight.detach().float().contiguous()
        n_out, k = w.shape
        (dyd, dyc), (xd, xc) = _mat(dy), _mat(xs[i])
        dw, _ = grads.get(lin.weight); db, _ = grads.get(lin.bias)
        sgemm(dyd, dyc, 1, n_out, xd, xc, k, 1, n_out, k, m, dw, F32, k)
        colsum(dyd, dyc, m, n_out, n_out, db)
        if i == 0 and dx is None:
            break
        dxi = dx if i == 0 else _f32((m, k), w.device)
        mask = xd if i > 0 and chain[i - 1][1] else None
        dxd, dxc = _mat(dxi)
        sgemm(dyd, dyc, n_out, 1, w, F32, k, 1, m, k, n_out, dxd, dxc, k, mask=mask,
              mask_ld=0 if mask is None else k)
        dy = dxi
    if isinstance(dx, Activation):
        dx.refresh_split()
    return dx


def encoder_forward_train(enc, inp: torch.Tensor, prec: str, bias3_host: torch.Tensor, width: int = 512):
    """node_encoder / edge_encoder (Models/BuckGNN.py:68-82): the two narrow Linears on bg_sgemm (fp32), the
    128 -> 512 one on the tensor cores.  Returns (h1 [n,64] f32, h2 [n,128], out [n,512]).
    width 128: the 2-layer encoder Linear(F,64) ReLU Linear(64,128) (:41-48), both on bg_sgemm; returns
    (h1 [n,64] f32, None, out [n,128])."""
    dev, n = inp.device, inp.shape[0]
    with engine.TIMERS.span("train_encoder"):
        h = Activation(n, 128, prec, dev)                    # h2, or the output at width 128
        _, (_, h1) = chain_forward(_linears(enc)[:2], inp, out=h)
        if width == 128:
            return h1, None, h
        out = Activation(n, 512, prec, dev)
        engine.gemm512(engine._segments(h, engine.pack_linear(enc[4].weight, prec)), n, prec, out,
                       bias=bias3_host.data_ptr())
    return h1, h, out


def encoder_backward(enc, inp: torch.Tensor, h1: torch.Tensor, h2: Optional[Activation], dout: Activation, prec: str,
                     grads: GradStore) -> None:
    """Gradients of the three encoder Linears given d(out) [n, 512] (of the two given d(out) [n, 128] at width 128,
    where h2 is None)."""
    dev, n = inp.device, inp.shape[0]
    code = engine.PRECISION_FORMATS[prec][0]
    s = _stream()
    with engine.TIMERS.span("train_encoder_bwd"):
        dh = dout                                                 # d(output of the bg_sgemm Linears)
        if h2 is not None:
            w3 = enc[4].weight.detach().float().contiguous()      # [512, 128]
            dw3e, _ = grads.get(enc[4].weight); db3e, _ = grads.get(enc[4].bias)
            tmp = _f32((512, 512), dev)
            weight_grad_mn(dout.data, h2.data, code, n, tmp, False)    # dW3 = dout^T h2; columns >= 128 of tmp come out 0
            dw3e.copy_(tmp[:, :128])
            colsum(dout.data, code, n, 512, 512, db3e)
            # dh2 = (dout W3) [h2 > 0]: W3^T zero-padded to 512 output rows on the tensor cores, then mask + narrow
            w3t_pad = torch.zeros((512, 512), dtype=torch.float32, device=dev)
            capi.transpose_chunks(w3.data_ptr(), capi.BG_F32, 512, 128, 128, 1, 512, w3t_pad.data_ptr(), s)
            full = Activation(n, 512, prec, dev)
            engine.gemm512(engine._segments(dout, engine.pack_linear(w3t_pad, prec)), n, prec, full)
            dh = _f32((n, 128), dev)
            capi.mask_narrow(full.data.data_ptr(), code, 512, h2.data.data_ptr(), code, 128, n, 128, dh.data_ptr(), s)
        chain_backward(_linears(enc)[:2], [inp, h1], dh, grads)


def _keep_head(sv, chain, xs, mlp: bool) -> None:
    """The head's chain and the input of each of its Linears for the backward pass.  The decoder's input and hidden
    layers are also kept by name: dec_in, h1d and h2d (None for the 2-layer decoder of h <= 128); `mlp` is MLPPooling's
    Linear, or None."""
    sv.head, sv.head_in = chain, xs
    sv.mlp = chain[0][0] if mlp else None
    sv.dec_in, sv.h1d, *h2d = xs[int(mlp):]
    sv.h2d = h2d[0] if h2d else None


def head_forward_train(model, cur: Activation, idx, sv) -> torch.Tensor:
    """get_pooling_layer + decoder (Models/BuckGNN.py:246-307, 515-516): the pooled feature comes from bg_pool_head
    (its own decoder output is not used here); MLPPooling (:568-581) and the decoder run on bg_sgemm so that their
    hidden layers are kept for the backward pass."""
    mlp = model.pooling_layer in ("mlp", "mlp_no_super")
    chain = (_linears(model.pooling_mpl.mlp) if mlp else []) + _linears(model.decoder)
    with engine.TIMERS.span("pool_head"):
        _, raw = engine.pool_head(cur, idx, engine.pack_decoder(model.decoder, cur.data.shape[1]), model.output_dim,
                                  want_pooled=True, pooling=model.pooling_layer)
        pred, xs = chain_forward(chain, raw)
    _keep_head(sv, chain, xs, mlp)
    return pred


def head_backward(model, sv, dpred: torch.Tensor, n: int, prec: str, grads: GradStore) -> Activation:
    """Decoder (+ MLPPooling) and pooling backward: returns d(last layer output) [n, hidden_channels]."""
    dev, W = dpred.device, model.hidden_channels
    g_count, in_dim = sv.head_in[0].shape
    with engine.TIMERS.span("train_head_bwd"):
        dpooled = chain_backward(sv.head, sv.head_in, dpred, grads, dx=_f32((g_count, in_dim), dev))
        dcur = Activation(n, W, prec, dev)
        capi.pool_backward(dpooled.data_ptr(), in_dim, sv.idx.graph_ptr.data_ptr(), g_count,
                           capi.POOL_MODES[model.pooling_layer], n, dcur.data.data_ptr(), dcur.code, _stream(), width=W)
    return dcur


def is_node_level(model) -> bool:
    return "static" in model.prediction_type or "mode_shape" in model.prediction_type


def node_head_forward_train(model, cur: Activation, sv) -> torch.Tensor:
    """Node-level heads (`static_disp`, `static_stress`, `mode_shape`): `decoder(x)` on every node
    (Models/BuckGNN.py:518-524; the caller drops the super-node rows) on bg_sgemm, its hidden layers kept for the
    backward pass."""
    if len(model.decoder) != 5 and not model._runs_native128_node_head():
        raise NotImplementedError("buckgnn_b200: node-level training needs the 3-layer decoder (hidden_channels >= 256), "
                                  "or hidden_channels = 128 with native128_node_head on")
    chain = _linears(model.decoder)
    with engine.TIMERS.span("node_head"):
        pred, xs = chain_forward(chain, cur)
    _keep_head(sv, chain, xs, False)
    return pred


def node_head_backward(model, sv, dpred: torch.Tensor, n: int, prec: str, grads: GradStore) -> Activation:
    """Backward of `decoder(x)` over all n nodes: returns d(last layer output) [n, hidden_channels]."""
    with engine.TIMERS.span("train_head_bwd"):
        return chain_backward(sv.head, sv.head_in, dpred, grads,
                              dx=Activation(n, model.hidden_channels, prec, dpred.device))


# ----------------------------------------------------------------------------- GraphSAGE
class SageTrainFunction(torch.autograd.Function):
    """pred = f(parameters); x / edge_index / batch are data (no gradient)."""

    @staticmethod
    def forward(ctx, model, x, edge_index, batch, seed, *params):
        prec = model.train_precision
        code = engine.PRECISION_FORMATS[prec][0]
        dev = x.device
        s = _stream()
        x = x.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        W = model.hidden_channels                          # 512, or 128 (BuckGNN.native128_train)
        if W not in (512, 128):
            raise NotImplementedError(f"buckgnn_b200: the training step runs at width 512 or 128, not {W}")
        if W == 128 and is_node_level(model) and not model._runs_native128_node_head():
            raise NotImplementedError("buckgnn_b200: the 128-wide training step has node-level heads only with "
                                      "native128_node_head on")
        convs = model._sage_layers()
        L = len(convs)
        aggr = convs[0][0].aggr if convs else "mean"      # no layers: the default model_name (encoder -> pool -> decoder)
        p_drop = float(model.dropout.p)
        pending = engine.begin_graph_index(edge_index, batch, n)
        # one read-back for all epilogue bias vectors of the step (they travel as kernel parameters)
        enc = model.node_encoder
        uniq_convs = []
        for c, _ in convs:
            if all(c is not q for q in uniq_convs):
                uniq_convs.append(c)
        biases = torch.stack([enc[-1].bias.detach().float()] + [c.lin_l.bias.detach().float() for c in uniq_convs]).cpu()
        bias_of = {id(c): biases[1 + k] for k, c in enumerate(uniq_convs)}

        sv = _Saved()
        sv.model, sv.prec, sv.n, sv.x, sv.seed, sv.p_drop, sv.aggr = model, prec, n, x, seed, p_drop, aggr
        sv.h1, sv.h2, cur = encoder_forward_train(enc, x, prec, biases[0], width=W)  # Models/BuckGNN.py:323
        idx = pending.finish()
        sv.idx = idx
        sv.edge_index = pending.edge_index
        # ---- layers
        packs = {}
        sv.layers = []
        ws_bytes = capi.train_workspace_bytes(n)
        ws = _ws(ws_bytes, dev)
        ones = torch.ones(W, dtype=torch.float32, device=dev)
        zeros = torch.zeros(W, dtype=torch.float32, device=dev)
        for i, (conv, bn) in enumerate(convs):
            if id(conv) not in packs:
                packs[id(conv)] = (engine.pack_linear(conv.lin_l.weight, prec), engine.pack_linear(conv.lin_r.weight, prec))
            wl, wr = packs[id(conv)]
            agg = Activation(n, W, prec, dev)
            engine.aggregate(cur, agg, idx, aggr)
            u = Activation(n, W, prec, dev)
            inv_norm = _f32((n,), dev)
            with engine.TIMERS.span("train_update_gemm"):
                engine.gemm(engine._segments(agg, wl) + engine._segments(cur, wr), n, prec, u,
                            bias=bias_of[id(conv)].data_ptr(), normalize=True, inv_norm_out=inv_norm.data_ptr())
            vec = None
            if bn is not None:
                vec = _f32((4, W), dev)                # a, shift, mean, invstd
                track = bn.track_running_stats and bn.running_mean is not None
                momentum = 0.1 if bn.momentum is None else float(bn.momentum)
                with engine.TIMERS.span("train_bn_stats"):
                    capi.bn_batch_stats(u.data.data_ptr(), code, n, bn.weight.detach().data_ptr(), bn.bias.detach().data_ptr(),
                                        float(bn.eps), momentum, bn.running_mean.data_ptr() if track else None,
                                        bn.running_var.data_ptr() if track else None,
                                        bn.num_batches_tracked.data_ptr() if track else None,
                                        vec[0].data_ptr(), vec[1].data_ptr(), vec[2].data_ptr(), vec[3].data_ptr(),
                                        ws.data_ptr(), ws_bytes, s, width=W)
                a_vec, shift_vec = vec[0], vec[1]
            else:
                a_vec, shift_vec = ones, zeros
            residual = 0 < i < L - 1
            y = Activation(n, W, prec, dev)
            with engine.TIMERS.span("train_bn_act"):
                capi.bn_act_forward(u.data.data_ptr(), cur.data.data_ptr() if residual else None, y.data.data_ptr(), code, n,
                                    a_vec.data_ptr(), shift_vec.data_ptr(), p_drop, layer_seed(seed, i), s, width=W)
            y.refresh_split()
            sv.layers.append((conv, bn, cur, agg, u, inv_norm, vec, residual))
            cur = y
        sv.ones, sv.zeros = ones, zeros
        sv.node_level = is_node_level(model)
        pred = node_head_forward_train(model, cur, sv) if sv.node_level else head_forward_train(model, cur, idx, sv)
        ctx.sv = sv
        ctx.params = trainable_parameters(model)      # the module's own parameters key the GradStore (the inputs may be embeddings, narrow.py)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        sv = ctx.sv
        model, prec, n = sv.model, sv.prec, sv.n
        code = engine.PRECISION_FORMATS[prec][0]
        dev = sv.x.device
        s = _stream()
        dpred = dpred.detach().to(torch.float32).contiguous()
        grads = GradStore(dev, getattr(model, "_grad_sync", None))
        dcur = (node_head_backward if sv.node_level else head_backward)(model, sv, dpred, n, prec, grads)
        grads.done(_head_params(model))                      # decoder (+ MLPPooling): their all-reduce starts now
        first_use = {}
        for j, (c_, _b, *_rest) in enumerate(sv.layers):
            first_use.setdefault(id(c_), j)                  # a shared block is final after its first (last visited) layer
        dy2: Optional[Activation] = None

        # ---- message passing layers, last to first
        idx = sv.idx
        idx_t = engine.build_graph_index(sv.edge_index, None, n, key_row=0) if sv.layers else None   # A^T
        ws_bytes = capi.train_workspace_bytes(n)
        ws = _ws(ws_bytes, dev)
        tpacks = {}
        mean = sv.aggr == "mean"
        L = len(sv.layers)
        W = model.hidden_channels
        for i in range(L - 1, -1, -1):
            conv, bn, x_in, agg, u, inv_norm, vec, residual = sv.layers[i]
            dz = Activation(n, W, prec, dev)
            dzs = Activation(n, W, prec, dev) if mean else dz
            g = Activation(n, W, prec, dev) if residual else None
            if bn is not None:
                dgam, acc_g = grads.get(bn.weight); dbet, _ = grads.get(bn.bias)
                a_vec, shift_vec, mean_vec, invstd_vec = vec[0], vec[1], vec[2], vec[3]
            else:
                dgam = dbet = mean_vec = invstd_vec = None
                acc_g = False
                a_vec, shift_vec = sv.ones, sv.zeros
            with engine.TIMERS.span("train_bwd_rows"):
                capi.sage_backward_rows(u.data.data_ptr(), dcur.data.data_ptr(), None if dy2 is None else dy2.data.data_ptr(),
                                        inv_norm.data_ptr(), idx.rowptr.data_ptr() if mean else None, code, n,
                                        a_vec.data_ptr(), shift_vec.data_ptr(), _p(mean_vec), _p(invstd_vec), sv.p_drop,
                                        layer_seed(sv.seed, i), _p(dgam), _p(dbet), acc_g, dz.data.data_ptr(),
                                        dzs.data.data_ptr() if mean else None, None if g is None else g.data.data_ptr(),
                                        ws.data_ptr(), ws_bytes, s, width=W)
            dz.refresh_split()
            if mean:
                dzs.refresh_split()
            # weight gradients: split over nodes on the tensor cores, operands read where they lie (MN-major)
            with engine.TIMERS.span("train_wgrad"):
                dwl, acc_l = grads.get(conv.lin_l.weight)
                dwr, acc_r = grads.get(conv.lin_r.weight)
                sage_weight_grads(dz.data, agg.data, x_in.data, code, n, dwl, acc_l, dwr, acc_r)
                dbl, acc_b = grads.get(conv.lin_l.bias)
                colsum(dz.data, code, n, W, W, dbl, accumulate=acc_b)
            # input gradient: dx = dz Wr + A^T (dz/deg Wl)  (+ g, added by the next iteration through dy2)
            if id(conv) not in tpacks:
                tpacks[id(conv)] = (transposed_pack(conv.lin_l.weight, prec), transposed_pack(conv.lin_r.weight, prec))
            wlt, wrt = tpacks[id(conv)]
            dagg = Activation(n, W, prec, dev)
            with engine.TIMERS.span("train_dgrad_gemm"):
                engine.gemm(engine._segments(dzs, wlt), n, prec, dagg)
            sbuf = Activation(n, W, prec, dev)
            if sv.aggr == "max":                     # the gradient goes to the neighbours that attain the maximum
                wtmp = Activation(n, W, prec, dev)
                mb = capi.max_bwd_workspace_bytes(idx.n_big, idx_t.n_big)
                mws = _ws(mb, dev)
                with engine.TIMERS.span("train_max_bwd"):
                    capi.max_aggregate_backward(x_in.data.data_ptr(), agg.data.data_ptr(), dagg.data.data_ptr(), code, n,
                                                idx.rowptr.data_ptr(), idx.col.data_ptr(), idx.big_rows.data_ptr(), idx.n_big,
                                                idx_t.rowptr.data_ptr(), idx_t.col.data_ptr(), idx_t.big_rows.data_ptr(),
                                                idx_t.n_big, wtmp.data.data_ptr(), sbuf.data.data_ptr(), mws.data_ptr(), mb, s,
                                                width=W)
                sbuf.refresh_split()
            else:
                engine.aggregate(dagg, sbuf, idx_t, "sum")
            dx = Activation(n, W, prec, dev)
            with engine.TIMERS.span("train_dgrad_gemm"):
                engine.gemm(engine._segments(dz, wrt), n, prec, dx, residual=sbuf.data.data_ptr(), ldr=W)
            if first_use[id(conv)] == i:
                grads.done([conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight] +
                           ([bn.weight, bn.bias] if bn is not None else []))
            dcur, dy2 = dx, g
        # ---- encoder backward (dy2 is None here: layer 0 has no skip)
        encoder_backward(model.node_encoder, sv.x, sv.h1, sv.h2, dcur, prec, grads)
        grads.finish()
        ctx.sv = None
        return (None, None, None, None, None, *grads.for_params(ctx.params))


# ----------------------------------------------------------------------------- GraphSAGE_SAG
def _sag_layer_forward(conv, bn, cur: Activation, idx, prec: str, bias_host, residual: bool, p_drop: float, seed_i: int,
                       ws, ws_bytes, ones, zeros):
    """One layer of the GraphSAGE_SAG loops (Models/BuckGNN.py:494-511): x = dropout(relu(bn(conv(x)))), then
    `x + identity` -- the skip is added AFTER the dropout here, unlike the plain variants."""
    dev, n = cur.data.device, cur.data.shape[0]
    code = cur.code
    s = _stream()
    wl, wr = engine.pack_linear(conv.lin_l.weight, prec), engine.pack_linear(conv.lin_r.weight, prec)
    agg = Activation(n, 512, prec, dev)
    engine.aggregate(cur, agg, idx, "add")
    u = Activation(n, 512, prec, dev)
    inv_norm = _f32((n,), dev)
    with engine.TIMERS.span("train_update_gemm"):
        engine.gemm512(engine._segments(agg, wl) + engine._segments(cur, wr), n, prec, u, bias=bias_host.data_ptr(),
                       normalize=True, inv_norm_out=inv_norm.data_ptr())
    vec = _f32((4, 512), dev)
    track = bn.track_running_stats and bn.running_mean is not None
    momentum = 0.1 if bn.momentum is None else float(bn.momentum)
    capi.bn_batch_stats(u.data.data_ptr(), code, n, bn.weight.detach().data_ptr(), bn.bias.detach().data_ptr(), float(bn.eps),
                        momentum, bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                        bn.num_batches_tracked.data_ptr() if track else None, vec[0].data_ptr(), vec[1].data_ptr(),
                        vec[2].data_ptr(), vec[3].data_ptr(), ws.data_ptr(), ws_bytes, s)
    y = Activation(n, 512, prec, dev)
    capi.bn_act_forward(u.data.data_ptr(), None, y.data.data_ptr(), code, n, vec[0].data_ptr(), vec[1].data_ptr(), p_drop, seed_i, s)
    if residual:
        capi.add(y.data.data_ptr(), cur.data.data_ptr(), None, y.data.data_ptr(), code, y.data.numel(), s)
    y.refresh_split()
    return y, (conv, bn, cur, agg, u, inv_norm, vec, residual, seed_i)


def _sag_layer_backward(saved, gup: Activation, idx, idx_t, prec: str, p_drop: float, grads: GradStore, ws, ws_bytes) -> Activation:
    """Backward of `_sag_layer_forward`: `gup` is d loss / d (layer output); returns d loss / d (layer input)."""
    conv, bn, x_in, agg, u, inv_norm, vec, residual, seed_i = saved
    dev, n = gup.data.device, gup.data.shape[0]
    code = gup.code
    s = _stream()
    dz = Activation(n, 512, prec, dev)
    dgam, acc_g = grads.get(bn.weight); dbet, _ = grads.get(bn.bias)
    capi.sage_backward_rows(u.data.data_ptr(), gup.data.data_ptr(), None, inv_norm.data_ptr(), None, code, n,
                            vec[0].data_ptr(), vec[1].data_ptr(), vec[2].data_ptr(), vec[3].data_ptr(), p_drop, seed_i,
                            dgam.data_ptr(), dbet.data_ptr(), acc_g, dz.data.data_ptr(), None, None, ws.data_ptr(), ws_bytes, s)
    dz.refresh_split()
    dwl, acc_l = grads.get(conv.lin_l.weight)
    dwr, acc_r = grads.get(conv.lin_r.weight)
    weight_grad_mn(dz.data, agg.data, code, n, dwl, acc_l)
    weight_grad_mn(dz.data, x_in.data, code, n, dwr, acc_r)
    dbl, acc_b = grads.get(conv.lin_l.bias)
    colsum(dz.data, code, n, 512, 512, dbl, accumulate=acc_b)
    wlt, wrt = transposed_pack(conv.lin_l.weight, prec), transposed_pack(conv.lin_r.weight, prec)
    dagg = Activation(n, 512, prec, dev)
    engine.gemm512(engine._segments(dz, wlt), n, prec, dagg)
    sbuf = Activation(n, 512, prec, dev)
    engine.aggregate(dagg, sbuf, idx_t, "sum")                      # A^T dagg ('add' aggregation: no degree scaling)
    dx = Activation(n, 512, prec, dev)
    engine.gemm512(engine._segments(dz, wrt), n, prec, dx, residual=sbuf.data.data_ptr(), ldr=512)
    if residual:                                                    # the skip branch carries the undropped gradient
        capi.add(dx.data.data_ptr(), gup.data.data_ptr(), None, dx.data.data_ptr(), code, dx.data.numel(), s)
        dx.refresh_split()
    return dx


class SagTrainFunction(torch.autograd.Function):
    """Training step of `GraphSAGE_SAG` (Models/BuckGNN.py:190-217, 493-511): num_layers // 2 SAGE('add') layers,
    SAGPooling(0.5) -- differentiable through `x[perm] * score[perm]` and the tanh score GNN, the selection itself is
    piecewise constant -- then the remaining layers on the pooled graph, pooling and the eigenvalue head."""

    @staticmethod
    def forward(ctx, model, x, edge_index, batch, seed, *params):
        prec = model.train_precision
        dev = x.device
        x = x.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        p_drop = float(model.dropout.p)
        pending = engine.begin_graph_index(edge_index, batch, n)
        enc = model.node_encoder
        convs = model._sage_layers()
        n_before = len(model.sage_layers_1)
        biases = torch.stack([enc[4].bias.detach().float()] + [c.lin_l.bias.detach().float() for c, _ in convs]).cpu()
        sv = _Saved()
        sv.model, sv.prec, sv.n, sv.x, sv.seed, sv.p_drop = model, prec, n, x, seed, p_drop
        sv.h1, sv.h2, cur = encoder_forward_train(enc, x, prec, biases[0])
        idx = pending.finish()
        sv.idx_full, sv.edge_index = idx, pending.edge_index
        ws_bytes = capi.train_workspace_bytes(n)
        ws = _ws(ws_bytes, dev)
        ones = torch.ones(512, dtype=torch.float32, device=dev)
        zeros = torch.zeros(512, dtype=torch.float32, device=dev)
        sv.first, sv.second = [], []
        for i in range(n_before):
            conv, bn = convs[i]
            cur, saved = _sag_layer_forward(conv, bn, cur, idx, prec, biases[1 + i], i > 0, p_drop, layer_seed(seed, i),
                                            ws, ws_bytes, ones, zeros)
            sv.first.append(saved)
        sv.pool_in = cur
        pack = engine.pack_sag_pool(model.pool)
        pooled = engine.sag_pool(cur, idx, idx.graph_ptr, idx.n_graphs, edge_index, pack, sign=model._sag_sign)
        model.last_pool = engine.pool_summary(pooled)   # perm / score / edge_index / batch of the last pooling, without its feature rows
        sv.pooled, sv.pool_pack = pooled, pack
        idx2 = engine.build_graph_index(pooled.edge_index, pooled.batch, pooled.n_nodes)
        sv.idx = idx2                                   # head_backward reads sv.idx.graph_ptr
        cur = pooled.x
        for k in range(n_before, len(convs)):
            conv, bn = convs[k]
            cur, saved = _sag_layer_forward(conv, bn, cur, idx2, prec, biases[1 + k], True, p_drop, layer_seed(seed, k),
                                            ws, ws_bytes, ones, zeros)
            sv.second.append(saved)
        pred = head_forward_train(model, cur, idx2, sv)
        ctx.sv = sv
        ctx.params = trainable_parameters(model)      # the module's own parameters key the GradStore (the inputs may be embeddings, narrow.py)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        sv = ctx.sv
        model, prec, n = sv.model, sv.prec, sv.n
        code = engine.PRECISION_FORMATS[prec][0]
        dev = sv.x.device
        s = _stream()
        F32 = capi.BG_F32
        grads = GradStore(dev, getattr(model, "_grad_sync", None))
        pooled, idx2 = sv.pooled, sv.idx
        n2 = pooled.n_nodes
        dcur = head_backward(model, sv, dpred.detach().to(torch.float32).contiguous(), n2, prec, grads)
        ws_bytes = capi.train_workspace_bytes(n)
        ws = _ws(ws_bytes, dev)
        if sv.second:
            idx2_t = engine.build_graph_index(pooled.edge_index, None, n2, key_row=0)
            for saved in reversed(sv.second):
                dcur = _sag_layer_backward(saved, dcur, idx2, idx2_t, prec, sv.p_drop, grads, ws, ws_bytes)
        # ---- SAGPooling backward
        idx_t = engine.build_graph_index(sv.edge_index, None, n, key_row=0)
        xin = sv.pool_in
        dx = Activation(n, 512, prec, dev)
        t, dpre = _f32((n,), dev), _f32((n,), dev)
        pack = sv.pool_pack
        with engine.TIMERS.span("sag_pool_bwd"):
            capi.sag_pool_backward(dcur.data.data_ptr(), xin.data.data_ptr(), code, n, n2, pooled.perm.data_ptr(),
                                   pooled.new_id.data_ptr(), pooled.all_scores.data_ptr(), float(model._sag_sign),
                                   idx_t.rowptr.data_ptr(), idx_t.col.data_ptr(), idx_t.big_rows.data_ptr(), idx_t.n_big,
                                   pack["w_l"].data_ptr(), pack["w_r"].data_ptr(), dx.data.data_ptr(), t.data_ptr(),
                                   dpre.data_ptr(), s)
            dx.refresh_split()
            gnn = model.pool.gnn
            dwl, _ = grads.get(gnn.lin_l.weight); dwr, _ = grads.get(gnn.lin_r.weight); dbl, _ = grads.get(gnn.lin_l.bias)
            # dw_l = sum_j t_j x_j, dw_r = sum_j dpre_j x_j: [1, n] x [n, 512]
            sgemm(t, F32, 0, 1, xin.data, code, 512, 1, 1, 512, n, dwl, F32, 512)
            sgemm(dpre, F32, 0, 1, xin.data, code, 512, 1, 1, 512, n, dwr, F32, 512)
            colsum(dpre, F32, n, 1, 1, dbl)
        dcur = dx
        for saved in reversed(sv.first):
            dcur = _sag_layer_backward(saved, dcur, sv.idx_full, idx_t, prec, sv.p_drop, grads, ws, ws_bytes)
        encoder_backward(model.node_encoder, sv.x, sv.h1, sv.h2, dcur, prec, grads)
        grads.finish()
        ctx.sv = None
        return (None, None, None, None, None, *grads.for_params(ctx.params))


def _head_params(model):
    ps = []
    if model.pooling_layer in ("mlp", "mlp_no_super") and not is_node_level(model):
        ps += [model.pooling_mpl.mlp[0].weight, model.pooling_mpl.mlp[0].bias]
    for m in model.decoder:
        if isinstance(m, torch.nn.Linear):
            ps += [m.weight, m.bias]
    return ps


def trainable_parameters(model) -> List[torch.nn.Parameter]:
    """Parameters the training step produces gradients for (the reference registers more modules than a given
    `model_name` uses: Models/BuckGNN.py:164,184-187)."""
    ps: List[torch.nn.Parameter] = []
    seen = set()

    def add(p):
        if p is not None and id(p) not in seen:
            seen.add(id(p)); ps.append(p)

    def add_seq(seq):
        for m in seq:
            if isinstance(m, torch.nn.Linear):
                add(m.weight); add(m.bias)

    add_seq(model.node_encoder)
    if model.model_name in ("EA_GNN", "EA_GNN_Shared", "EAGNN_SAG"):
        add_seq(model.edge_encoder)
        if model.model_name == "EAGNN_SAG":
            blocks = list(model.gnn_layers_1) + list(model.gnn_layers_2)
        else:
            blocks = [model.shared_gn_block] if model.model_name == "EA_GNN_Shared" else list(model.gn_blocks)
        for blk in blocks:
            for seq in (blk.edge_mlp, blk.node_mlp_phi, blk.node_mlp_gamma, blk.node_mlp_beta):
                add_seq(seq)
    for conv, bn in model._sage_layers():
        add(conv.lin_l.weight); add(conv.lin_l.bias); add(conv.lin_r.weight)
        if bn is not None:
            add(bn.weight); add(bn.bias)
    if model.model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):
        gnn = model.pool.gnn
        add(gnn.lin_l.weight); add(gnn.lin_l.bias); add(gnn.lin_r.weight)
    if model.pooling_layer in ("mlp", "mlp_no_super") and not is_node_level(model):
        add(model.pooling_mpl.mlp[0].weight); add(model.pooling_mpl.mlp[0].bias)
    add_seq(model.decoder)
    return ps


def forward_train(model, x, edge_index, batch, seed: Optional[int] = None, edge_attr=None) -> torch.Tensor:
    if seed is None:                                    # one draw from torch's generator per step, like nn.Dropout
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    params = trainable_parameters(model)
    inputs = getattr(model, "_param_inputs", None)
    if inputs:          # narrow.WideTwin: the twin's parameters as differentiable embeddings of the narrow model's
        params = [inputs.get(id(p_), p_) for p_ in params]
    if model.model_name in ("EA_GNN", "EA_GNN_Shared"):
        from .train_eagnn import EAGNNTrainFunction
        return EAGNNTrainFunction.apply(model, x, edge_index, edge_attr, batch, seed, *params)
    if model.model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):
        if is_node_level(model):
            raise NotImplementedError("buckgnn_b200: the SAGPooling variants train with the eigenvalue head only")
        if batch is None:
            batch = torch.zeros(x.shape[0], dtype=torch.int64, device=x.device)
        if model.model_name == "EAGNN_SAG":
            from .train_eagnn import EAGNNSagTrainFunction
            return EAGNNSagTrainFunction.apply(model, x, edge_index, edge_attr, batch, seed, *params)
        return SagTrainFunction.apply(model, x, edge_index, batch, seed, *params)
    return SageTrainFunction.apply(model, x, edge_index, batch, seed, *params)
