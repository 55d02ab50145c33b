"""`BuckGNN` with the reference's module contract, running on the sm_100a kernels.

Mirrors `Models/BuckGNN.py` of the reference:
  * constructor arguments, attribute names and parameter registration order
    (`:10-244`) -> identical `state_dict()` keys and shapes, so checkpoints written
    by `TRAIN_FINAL.py:394-410` load with `strict=True`;
  * `forward(x, edge_index, edge_attr, batch=None, mask=None)` -> `(pred, batch)`
    (`:311`, `:516`); `pred` is `[G]` after `.squeeze()` (0-dim when G == 1), the
    second element is the caller's `batch` object unchanged;
  * errors: `ValueError("Unknown pooling layer: ...")` (`:307`) and
    `ValueError("Unknown prediction type: ...")` (`:526`).

The forward never touches PyG / torch_scatter / ATen math: it is the kernel sequence
in `engine.py`.  CPU tensors raise -- there is no fallback path.

In train mode (`model.train()`, as TRAIN_FINAL.py:289 does) the forward uses batch statistics in
BatchNorm1d, applies Dropout and is differentiable: `loss.backward()` runs the backward kernels
(`train.py`) and leaves `.grad` on the parameters that model_name uses.

A hidden_channels = 128 GraphSAGE model (the reference's default width) evaluates on its own 128-wide kernels.  It
trains on them too when `model.native128_train` is set (a module attribute, default from BUCKGNN_NATIVE128_TRAIN=1 in
the environment); otherwise, and for what the 128-wide step does not cover, training runs as the zero-padded 512-wide
twin (narrow.py).  A 128-wide EA_GNN / EA_GNN_Shared model evaluates on the 128-wide kernels when
`model.native128_eagnn` is set (default from BUCKGNN_NATIVE128_EAGNN=1), and trains on them when
`model.native128_eagnn_train` is set (default from BUCKGNN_NATIVE128_EAGNN_TRAIN=1; train_eagnn.py at width 128);
otherwise it trains as the twin.  Those flags cover graph-level heads.  Node-level heads (static_disp, static_stress,
mode_shape) of the same eight models at 128 evaluate and train on the 128-wide kernels when `model.native128_node_head`
is set (default from BUCKGNN_NATIVE128_NODE_HEAD=1; bg_node_head128 in eval), and otherwise run as the twin.  The
SAGPooling variants and widths 64 / 256 always run as the twin.

Extra, non-reference keywords: `train_precision` in {"tf32", "bf16", "fp16"} (storage of the training
step's activations and activation gradients; default tf32 = fp32 storage), and `precision` in {"auto", "fp16", "bf16", "tf32", "fp32"}
selects how the tensor-core GEMMs read their operands (engine.PRECISION_FORMATS; fp32 =
3xTF32 split, the "fp32-GEMM mode"; "auto" = fp16 for mean/max aggregation, tf32 for
sum/add whose hub rows can leave the fp16 range).
"""
from __future__ import annotations

from typing import Dict, Optional

import os

import torch
import torch.nn as nn

from . import engine
from .engine import Activation, LinearPack, SageLayerPack

_SAGE_LISTS = {  # model_name -> (ModuleList attribute, aggr)      reference :120-180
    "GraphSage_sumAggr": ("sage_blocks_sum", "sum"),
    "GraphSage_addAggr": ("sage_blocks_add", "add"),
    "GraphSage_meanAggr": ("sage_blocks_mean", "mean"),
    "GraphSage_maxAggr": ("sage_blocks_max", "max"),
}
_POOLINGS = ("mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super")
# models whose eval forward at hidden_channels == 128 runs on the 128-wide kernels (the rest use narrow.WideTwin)
_NATIVE128_MODELS = tuple(_SAGE_LISTS) + ("GraphSage_addAggr_Shared", "GraphSAGE_MLP")
# train-mode forwards of the same models at hidden_channels == 128 on the 128-wide kernels (train.py at width 128)
# instead of the twin.  Opt-in: BUCKGNN_NATIVE128_TRAIN=1 in the environment, or `model.native128_train = True`.
NATIVE128_TRAIN_DEFAULT = os.environ.get("BUCKGNN_NATIVE128_TRAIN", "0") not in ("", "0")
# EA-GNN models whose eval forward at hidden_channels == 128 runs on the 128-wide kernels (bg_gemm128_gathered for the
# edge GEMMs) instead of the twin.  Opt-in: BUCKGNN_NATIVE128_EAGNN=1 in the environment, or
# `model.native128_eagnn = True`.
_NATIVE128_EAGNN_MODELS = ("EA_GNN", "EA_GNN_Shared")
NATIVE128_EAGNN_DEFAULT = os.environ.get("BUCKGNN_NATIVE128_EAGNN", "0") not in ("", "0")
# train-mode forwards of the same EA-GNN models at hidden_channels == 128 on the 128-wide kernels (train_eagnn.py at
# width 128) instead of the twin.  Opt-in: BUCKGNN_NATIVE128_EAGNN_TRAIN=1 in the environment, or
# `model.native128_eagnn_train = True`.
NATIVE128_EAGNN_TRAIN_DEFAULT = os.environ.get("BUCKGNN_NATIVE128_EAGNN_TRAIN", "0") not in ("", "0")
# node-level heads (static_disp, static_stress, mode_shape) of the models above at hidden_channels == 128: eval forward
# and training step on the 128-wide kernels (bg_node_head128 in eval, bg_sgemm in training) instead of the twin.
# Opt-in: BUCKGNN_NATIVE128_NODE_HEAD=1 in the environment, or `model.native128_node_head = True`.
NATIVE128_NODE_HEAD_DEFAULT = os.environ.get("BUCKGNN_NATIVE128_NODE_HEAD", "0") not in ("", "0")


class SAGEConv(nn.Module):
    """Parameter container with PyG SAGEConv's names: lin_l.{weight,bias}, lin_r.weight."""

    def __init__(self, in_channels: int, out_channels: int, normalize: bool = True, aggr: str = "mean"):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.normalize, self.aggr = normalize, aggr
        self.lin_l = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, *a, **k):  # pragma: no cover - the layer only runs fused inside BuckGNN.forward
        raise RuntimeError("buckgnn_b200.SAGEConv holds parameters only; it runs fused inside BuckGNN.forward")


def _mlp2(i, h, o):
    return nn.Sequential(nn.Linear(i, h), nn.ReLU(), nn.Linear(h, o))


class GraphNetBlock(nn.Module):
    """Parameter container for the reference's EA-GNN block (`:528-550`)."""

    def __init__(self, hidden_channels: int):
        super().__init__()
        h = hidden_channels
        self.edge_mlp = _mlp2(3 * h, h, h)
        self.node_mlp_phi = _mlp2(2 * h, h, h)
        self.node_mlp_gamma = _mlp2(2 * h, h, h)
        self.node_mlp_beta = _mlp2(h, h, h)


class MLPPooling(nn.Module):
    """Parameter container for the reference's `MLPPooling` (`:568-576`)."""

    def __init__(self, in_channels, hidden_channels, out_channels):
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(in_channels, hidden_channels), nn.ReLU())


class SAGPooling(nn.Module):
    """Parameter container with PyG `SAGPooling`'s names (`pool.gnn.lin_l.{weight,bias}`, `pool.gnn.lin_r.weight`;
    reference `:203-208`, `:231-236`): the scoring GNN is `SAGEConv(in_channels, 1, aggr='add')`."""

    def __init__(self, in_channels: int, ratio: float = 0.5, aggr: str = "add"):
        super().__init__()
        self.in_channels, self.ratio = in_channels, ratio
        self.gnn = SAGEConv(in_channels, 1, normalize=False, aggr=aggr)


def _output_dim(prediction_type, use_z_coord, use_rotations):
    if prediction_type == "buckling":
        return 1
    if prediction_type == "static_disp":
        return {(True, True): 6, (True, False): 3, (False, True): 4, (False, False): 2}[
            (bool(use_z_coord), bool(use_rotations))]
    if prediction_type == "static_stress":
        return 3
    if prediction_type == "mode_shape":
        return 6 if use_rotations else 3
    raise NameError("output_dim")          # the reference leaves output_dim unbound here (:20-38)


class BuckGNN(nn.Module):
    def __init__(self, num_node_features, num_edge_features, hidden_channels=128,
                 num_layers=6, pooling_layer="mean", prediction_type="buckling",
                 use_z_coord=False, use_rotations=False, dropout_rate=0.1,
                 model_name="GraphSAGE_MLP", *, precision: str = "auto", cta_group: int = 2,
                 cache_index: bool = False, fold_encoder: bool = True, train_precision: str = "tf32",
                 fuse_pool: bool = True):
        super().__init__()
        self._ctor_kwargs = dict(num_node_features=num_node_features, num_edge_features=num_edge_features,
                                 hidden_channels=hidden_channels, num_layers=num_layers, pooling_layer=pooling_layer,
                                 prediction_type=prediction_type, use_z_coord=use_z_coord, use_rotations=use_rotations,
                                 dropout_rate=dropout_rate, model_name=model_name, precision=precision, cta_group=cta_group,
                                 cache_index=cache_index, fold_encoder=fold_encoder, train_precision=train_precision,
                                 fuse_pool=fuse_pool)
        if precision == "auto":
            aggr = _SAGE_LISTS[model_name][1] if model_name in _SAGE_LISTS else (
                "add" if model_name == "GraphSage_addAggr_Shared" else "mean")
            precision = engine.default_precision(aggr)
            # GraphSAGE_SAG defaults to the fp32-GEMM mode: it picks nodes by a discrete top-k on a score and multiplies
            # the survivors by it, which (through the BatchNorms that follow) makes the prediction ~10x more sensitive to
            # operand rounding than the plain variants (emulated tf32 operands in the fp32 oracle: 1.3e-3 .. 1e-2,
            # tests/test_oracle.py), beyond the 1e-3 parity bar; the 3xTF32 mode stays below 1e-4.  EAGNN_SAG has no
            # BatchNorm and shows no such amplification (same emulation: ~2e-5 even when the selection differs); it
            # runs with fp32 storage and tf32 operands so that 16-bit rounding does not perturb the score order.
            if model_name == "GraphSAGE_SAG":
                precision = "fp32"
            elif model_name == "EAGNN_SAG":
                precision = "tf32"
        if precision not in engine.PRECISIONS:
            raise ValueError(f"precision must be \"auto\" or one of {engine.PRECISIONS}")
        if train_precision not in ("tf32", "bf16", "fp16"):
            raise ValueError('train_precision must be one of "tf32", "bf16", "fp16"')
        self.train_precision = train_precision          # storage of activations / their gradients in train mode
        self.hidden_channels = hidden_channels
        self.prediction_type = prediction_type
        self.pooling_layer = pooling_layer
        self.num_layers = num_layers
        self.model_name = model_name
        self.precision = precision
        self.cta_group = cta_group
        self.cache_index = cache_index
        self.fold_encoder = fold_encoder      # fold node_encoder[4] into SAGE layer 0 (mean / sum / add aggregation)
        self.fuse_pool = fuse_pool            # last SAGE layer's epilogue sums its rows for the pooling layer (16-bit modes)
        self.fuse_aggregate = engine.FUSE_AGGREGATE_DEFAULT    # the aggregate operand gathered inside the update GEMM (opt-in)
        self.native128_train = NATIVE128_TRAIN_DEFAULT         # hidden_channels 128: train on the 128-wide kernels (opt-in)
        self.native128_eagnn = NATIVE128_EAGNN_DEFAULT         # hidden_channels 128: EA-GNN eval on the 128-wide kernels (opt-in)
        self.native128_eagnn_train = NATIVE128_EAGNN_TRAIN_DEFAULT   # hidden_channels 128: EA-GNN training on them (opt-in)
        self.native128_node_head = NATIVE128_NODE_HEAD_DEFAULT       # hidden_channels 128: node-level heads on them (opt-in)
        self.output_dim = output_dim = _output_dim(prediction_type, use_z_coord, use_rotations)
        h = hidden_channels
        cat_dec = pooling_layer == "supernode_with_pooling" and prediction_type == "buckling"
        if h <= 128:
            self.node_encoder = _mlp2(num_node_features, 64, h)
            self.edge_encoder = _mlp2(num_edge_features, 64, h)
            self.decoder = _mlp2(2 * h if cat_dec else h, 64, output_dim)
        elif h >= 256:
            self.node_encoder = nn.Sequential(nn.Linear(num_node_features, 64), nn.ReLU(),
                                              nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, h))
            self.edge_encoder = nn.Sequential(nn.Linear(num_edge_features, 64), nn.ReLU(),
                                              nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, h))
            self.decoder = nn.Sequential(nn.Linear(2 * h if cat_dec else h, 128), nn.ReLU(),
                                         nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, output_dim))
        if model_name == "EA_GNN_Shared":
            self.shared_gn_block = GraphNetBlock(h)
        if model_name == "EA_GNN":
            self.gn_blocks = nn.ModuleList([GraphNetBlock(h) for _ in range(num_layers)])
        if model_name == "GraphSage_addAggr_Shared":
            self.shared_graphsage_block = SAGEConv(h, h, normalize=True, aggr="add")
        if model_name in _SAGE_LISTS:
            attr, aggr = _SAGE_LISTS[model_name]
            blocks, bns, mlps = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
            setattr(self, attr, blocks)
            self.batch_norms = bns
            self.sage_mlps = mlps
            for _ in range(num_layers):
                blocks.append(SAGEConv(h, h, normalize=True, aggr=aggr))
                bns.append(nn.BatchNorm1d(h))
                mlps.append(nn.Linear(h, h))
        self.batch_norm = nn.BatchNorm1d(h)
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(p=dropout_rate)
        self.pooling_mpl = MLPPooling(h, h, h)
        if model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):                 # reference :190-244 (registered after pooling_mpl)
            n_before = num_layers // 2
            n_after = num_layers - n_before
            sage = model_name == "GraphSAGE_SAG"
            mk = (lambda: SAGEConv(h, h, normalize=True, aggr="add")) if sage else (lambda: GraphNetBlock(h))
            setattr(self, "sage_layers_1" if sage else "gnn_layers_1", nn.ModuleList([mk() for _ in range(n_before)]))
            self.batch_norms_1 = nn.ModuleList([nn.BatchNorm1d(h) for _ in range(n_before)] if sage else [])
            self.pool = SAGPooling(h, ratio=0.5, aggr="add")
            setattr(self, "sage_layers_2" if sage else "gnn_layers_2", nn.ModuleList([mk() for _ in range(n_after)]))
            self.batch_norms_2 = nn.ModuleList([nn.BatchNorm1d(h) for _ in range(n_after)] if sage else [])
            # PyG >= 2.4 checkpoints carry `pool.select.weight` [1, 1]: SelectTopK multiplies the score by
            # weight / |weight| before tanh, i.e. by its sign.  Older ones (the formulation restated here) do not.
            self._sag_sign = 1.0
            self._register_load_state_dict_pre_hook(self._absorb_select_weight)
        self._packs: Dict[str, object] = {}
        self._pack_sig = None
        self._index_cache = None
        self._wide = None                     # hidden_channels != 512: the zero-padded 512-wide twin (narrow.py), built lazily
        self._ran_native128 = False           # the last forward ran on the 128-wide kernels (check_finite reads self)
        self._param_inputs = None             # set by narrow.WideTwin around a train-mode forward of the twin

    # ------------------------------------------------------------------ weight packing
    def _absorb_select_weight(self, state_dict, prefix, *args):
        key = prefix + "pool.select.weight"
        if key in state_dict:
            w = float(state_dict.pop(key).reshape(-1)[0])
            self._sag_sign = -1.0 if w < 0 else 1.0

    def _signature(self):
        return (self.precision, getattr(self, "_sag_sign", 1.0)) + tuple((p.data_ptr(), p._version) for p in self.parameters()) + \
            tuple((b.data_ptr(), b._version) for b in self.buffers())

    def _sage_layers(self):
        if self.model_name in _SAGE_LISTS:
            convs = getattr(self, _SAGE_LISTS[self.model_name][0])
            return [(c, bn) for c, bn in zip(convs, self.batch_norms)]
        if self.model_name == "GraphSage_addAggr_Shared":
            return [(self.shared_graphsage_block, None)] * self.num_layers
        if self.model_name == "GraphSAGE_SAG":
            return list(zip(self.sage_layers_1, self.batch_norms_1)) + list(zip(self.sage_layers_2, self.batch_norms_2))
        return []

    def _packed(self, width: int = 512):
        """Operand-format copies of the weights for the kernels of `width` (512, or 128: a hidden_channels = 128 model
        in eval on the 128-wide kernels), rebuilt when any parameter/buffer changes.  Only the encoders and the decoder
        pack differently at 128 (engine.pack_encoder / pack_decoder)."""
        sig = (width,) + self._signature()
        if self._pack_sig == sig:
            return self._packs
        prec = self.precision
        f32 = lambda t: t.detach().float().contiguous()
        enc = self.node_encoder
        packs = {}
        packs["enc"], packs["enc_w3"] = engine.pack_encoder(enc, prec, width)
        packs["dec"] = engine.pack_decoder(self.decoder, width)
        if self.prediction_type != "buckling" and self.hidden_channels >= 256:
            packs["node_head"] = engine.pack_node_head(self.decoder, prec)
        elif self.prediction_type != "buckling" and width == 128:
            packs["node_head"] = engine.pack_node_head128(self.decoder, prec)
        mpl = self.pooling_mpl.mlp[0]
        packs["pool_mlp"] = {"w": f32(mpl.weight), "b": f32(mpl.bias)}
        layers, seen = [], {}
        for conv, bn in self._sage_layers():
            if id(conv) not in seen:
                scale, shift = engine.fold_batchnorm(bn) if bn is not None else (None, None)
                seen[id(conv)] = SageLayerPack(engine.pack_linear(conv.lin_l.weight, prec),
                                               engine.pack_linear(conv.lin_r.weight, prec),
                                               engine.host_vector(conv.lin_l.bias), scale, shift)
            layers.append(seen[id(conv)])
        packs["layers"] = layers
        packs["layer0_folded"] = None
        sl = self._sage_layers()
        if self.model_name == "GraphSAGE_SAG" and len(self.sage_layers_1) == 0:
            sl = []                                   # num_layers == 1: the pooling runs on the encoder output itself
        if self.fold_encoder and sl and sl[0][0].aggr != "max":
            conv0, bn0 = sl[0]
            packs["layer0_folded"] = engine.pack_folded_layer0(enc[-1], conv0, bn0, conv0.aggr, prec,
                                                               width=width)                       # None: unfolded
        if self.model_name in ("EA_GNN", "EA_GNN_Shared", "EAGNN_SAG"):
            packs["edge_enc"], packs["edge_enc_w3"] = engine.pack_encoder(self.edge_encoder, prec, width)
        if self.model_name == "EA_GNN_Shared":
            packs["gn"] = [engine.pack_gnblock(self.shared_gn_block, prec, width=width)] * self.num_layers
        elif self.model_name == "EA_GNN":
            packs["gn"] = [engine.pack_gnblock(b, prec, width=width) for b in self.gn_blocks]
        if self.model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):
            packs["sag_pool"] = engine.pack_sag_pool(self.pool)
        if self.model_name == "EAGNN_SAG":
            packs["gn1"] = [engine.pack_gnblock(b, prec) for b in self.gnn_layers_1]
            packs["gn2"] = [engine.pack_gnblock(b, prec) for b in self.gnn_layers_2]
        self._packs, self._pack_sig = packs, sig
        return packs

    # ------------------------------------------------------------------ forward
    def _check_model_name(self):
        if self.model_name in ("GraphSage_MLP", "GraphSage_addAggr_woBatchNorm", "GraphSage_sumAggr_woBatchNorm"):
            # the reference constructs the module lists these branches use only under other names
            raise AttributeError(f"'BuckGNN' object has no module list for model_name={self.model_name!r} "
                                 "(same failure as the reference, Models/BuckGNN.py:404-429,472-492)")

    def _check_supported(self, x):
        self._check_model_name()
        if not x.is_cuda:
            raise RuntimeError("buckgnn_b200.BuckGNN runs on CUDA (sm_100a) tensors only; there is no CPU path")
        if self.hidden_channels > 512:
            raise NotImplementedError("buckgnn_b200: the tcgen05 path holds one 512-column row per TMEM lane; "
                                      "hidden_channels > 512 is not built")

    def _runs_native128(self) -> bool:
        """hidden_channels == 128 eval forwards of the GraphSAGE models with a graph-level head run on the 128-wide
        kernels, and those of EA_GNN / EA_GNN_Shared too when `native128_eagnn` is on; everything else at a width other
        than 512 runs on the zero-padded twin (narrow.py)."""
        if (self.hidden_channels != 128 or self.training or self.prediction_type != "buckling"
                or self.pooling_layer not in _POOLINGS):
            return False
        if self.model_name in _NATIVE128_EAGNN_MODELS:
            return bool(self.native128_eagnn)
        return not self.fuse_aggregate and self.model_name in _NATIVE128_MODELS

    def _trains_native128(self) -> bool:
        """With `native128_train` on, train-mode forwards of the models `_runs_native128` covers run the training step
        at width 128 on the module's own parameters (train.py); everything else at a width other than 512 trains as the
        twin, flag or no flag."""
        return (self.hidden_channels == 128 and self.training and bool(self.native128_train)
                and self.model_name in _NATIVE128_MODELS and self.prediction_type == "buckling"
                and self.pooling_layer in _POOLINGS)

    def _trains_native128_eagnn(self) -> bool:
        """With `native128_eagnn_train` on, train-mode forwards of EA_GNN / EA_GNN_Shared at hidden_channels == 128 with a
        graph-level head run the EA-GNN training step at width 128 on the module's own parameters (train_eagnn.py);
        `native128_train` and `native128_eagnn` leave them on the twin."""
        return (self.hidden_channels == 128 and self.training and bool(self.native128_eagnn_train)
                and self.model_name in _NATIVE128_EAGNN_MODELS and self.prediction_type == "buckling"
                and self.pooling_layer in _POOLINGS)

    def _runs_native128_node_head(self, training: Optional[bool] = None) -> bool:
        """With `native128_node_head` on, eval and train-mode forwards of the GraphSAGE models `_runs_native128` covers
        and of EA_GNN / EA_GNN_Shared at hidden_channels == 128 with a node-level head (static_disp, static_stress,
        mode_shape) run on the 128-wide kernels; the other three flags leave them on the twin.  GraphSAGE eval needs
        `fuse_aggregate` off, as in `_runs_native128`.  `training` overrides the module's mode."""
        training = self.training if training is None else training
        if (self.hidden_channels != 128 or not self.native128_node_head
                or not ("static" in self.prediction_type or "mode_shape" in self.prediction_type)):
            return False
        if self.model_name in _NATIVE128_EAGNN_MODELS:
            return True
        return self.model_name in _NATIVE128_MODELS and (training or not self.fuse_aggregate)

    def forward(self, x, edge_index, edge_attr, batch=None, mask=None):
        self._check_supported(x)
        self._ran_native128 = False
        if self._runs_native128_node_head():
            if self.training:
                from . import train
                pred = train.forward_train(self, x, edge_index, batch, edge_attr=edge_attr)
                self._pack_sig = None            # BatchNorm statistics changed: the next native eval forward repacks
            else:
                with torch.no_grad():
                    if self.model_name in _NATIVE128_EAGNN_MODELS:
                        pred = self._forward_cuda_eagnn(x, edge_index, edge_attr, batch, node_level=True, width=128)
                    else:
                        pred = self._forward_cuda(x, edge_index, batch, node_level=True, width=128)
                self._ran_native128 = True
            if "super" in self.pooling_layer:                # reference :518-524, as the twin returns it
                is_real_node = x[:, -1] == 0
                return pred[is_real_node], (batch[is_real_node] if batch is not None else None)
            return pred, batch
        if self._runs_native128():
            with torch.no_grad():
                if self.model_name in _NATIVE128_EAGNN_MODELS:
                    pred = self._forward_cuda_eagnn(x, edge_index, edge_attr, batch, width=128)
                else:
                    pred = self._forward_cuda(x, edge_index, batch, width=128)
            self._ran_native128 = True
            return pred.squeeze(), batch
        if self._trains_native128() or self._trains_native128_eagnn():
            from . import train
            pred = train.forward_train(self, x, edge_index, batch, edge_attr=edge_attr)
            self._pack_sig = None                # BatchNorm statistics changed: the next native eval forward repacks
            return pred.squeeze(), batch
        if self.hidden_channels != 512:
            if self.training and getattr(self, "_grad_sync", None) is not None:
                # the twin's parameters are not the module's own: the installed GradSync would never see a gradient
                raise NotImplementedError("buckgnn_b200: this model trains as the zero-padded 512-wide twin, which "
                                          "enable_gradient_sync does not cover; use dist.allreduce_gradients("
                                          "model.parameters()) after backward() instead")
            # TRAIN_FINAL.py:55,71 / the constructor default use 128: runs as the exact zero-padded 512-wide twin.
            # 129..255 build no encoder in the reference (Models/BuckGNN.py:41,67): the same AttributeError surfaces here.
            if self._wide is None:
                self.node_encoder                                    # AttributeError for 129 <= hidden <= 255, as the reference
                from .narrow import WideTwin
                self._wide = WideTwin(self, self._ctor_kwargs)
            out = self._wide.forward(x, edge_index, edge_attr, batch)
            if self.training:
                self._pack_sig = None            # BatchNorm statistics changed: the next native eval forward repacks
            return out
        node_level = "static" in self.prediction_type or "mode_shape" in self.prediction_type
        if self.prediction_type != "buckling" and not node_level:
            raise ValueError(f"Unknown prediction type: {self.prediction_type}")
        if node_level and self.hidden_channels < 256:
            raise NotImplementedError("buckgnn_b200: node-level heads need the 3-layer decoder (hidden_channels >= 256)")
        if not node_level and self.pooling_layer not in _POOLINGS:
            if self.pooling_layer == "hybrid":
                raise AttributeError("'BuckGNN' object has no attribute 'hybrid_pooling'")   # reference :188,276
            raise ValueError(f"Unknown pooling layer: {self.pooling_layer}")
        if self.training:       # train-mode BatchNorm / Dropout + autograd through the backward kernels (train.py)
            from . import train
            pred = train.forward_train(self, x, edge_index, batch, edge_attr=edge_attr)
            # the train-mode kernels update the BatchNorm running statistics through raw pointers (no version bump):
            # drop the eval-mode operand cache so the next eval forward folds the new statistics
            self._pack_sig = None
            if self.model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):   # `batch` was reassigned by self.pool (:365, :502)
                return pred.squeeze(), self.last_pool.batch
            if node_level:                                   # reference :518-524; the row selection is an autograd index
                if "super" in self.pooling_layer:
                    is_real_node = x[:, -1] == 0
                    return pred[is_real_node], (batch[is_real_node] if batch is not None else None)
                return pred, batch
            return pred.squeeze(), batch
        with torch.no_grad():
            if self.model_name in ("GraphSAGE_SAG", "EAGNN_SAG"):
                if node_level and "super" in self.pooling_layer:
                    # the reference indexes the POOLED x with the un-pooled is_real_node mask here (:518-521)
                    raise IndexError("The shape of the mask (is_real_node over all nodes) does not match the pooled node "
                                     "tensor (same failure as the reference, Models/BuckGNN.py:521 after SAGPooling)")
                fwd = self._forward_cuda_sag if self.model_name == "GraphSAGE_SAG" else self._forward_cuda_eagnn_sag
                pred, pooled_batch = fwd(x, edge_index, edge_attr, batch, node_level)
                return (pred if node_level else pred.squeeze()), pooled_batch      # `batch` was reassigned by self.pool (:365, :502)
            if self.model_name in ("EA_GNN", "EA_GNN_Shared"):
                pred = self._forward_cuda_eagnn(x, edge_index, edge_attr, batch, node_level)
            else:
                pred = self._forward_cuda(x, edge_index, batch, node_level)
        if node_level:                                       # reference :518-524
            if "super" in self.pooling_layer:
                is_real_node = x[:, -1] == 0                 # :315-320 (row selection of the [N, out] result)
                return pred[is_real_node], (batch[is_real_node] if batch is not None else None)
            return pred, batch
        return pred.squeeze(), batch

    def _new_nonfinite_flag(self, device):
        """Device word the 16-bit kernels raise when a value does not fit their storage format (bg_encoder_front);
        bg_pool_head turns it into NaN predictions.  Kept on the module for `check_finite()`."""
        self._nonfinite = torch.zeros(1, dtype=torch.int32, device=device)
        return self._nonfinite

    def enable_gradient_sync(self, group=None):
        """Multi-GPU training (BASELINE.json configs[3]): all-reduce (mean) the gradients of this model's trainable
        parameters over `group`, bucketed per layer and overlapped with the backward pass (dist.GradSync).  Call once
        after `.to(device)`, on every rank; `loss.backward()` then leaves the REDUCED gradients in `.grad`."""
        native128 = (self.native128_train or (self.native128_eagnn_train and self.model_name in _NATIVE128_EAGNN_MODELS)
                     or self._runs_native128_node_head(training=True))
        if self.hidden_channels != 512 and not (self.hidden_channels == 128 and native128):
            raise NotImplementedError("buckgnn_b200: overlapped gradient sync is built for hidden_channels=512, and for "
                                      "128 with native128_train (EA_GNN / EA_GNN_Shared: native128_eagnn_train; "
                                      "node-level heads: native128_node_head) on; use "
                                      "dist.allreduce_gradients(model.parameters()) after backward() instead")
        from . import train
        from .dist import GradSync
        self._grad_sync = GradSync(train.trainable_parameters(self), next(self.parameters()).device, group)
        return self._grad_sync

    def check_finite(self) -> None:
        """Raises FloatingPointError if the last eval-mode forward met activations its 16-bit storage format cannot
        hold (synchronises; the forward itself reports the condition as NaN predictions without a sync)."""
        target = self._wide.twin if self._wide is not None and not self._ran_native128 else self
        flag = getattr(target, "_nonfinite", None)
        if flag is not None and int(flag.item()) != 0:
            raise FloatingPointError(f"buckgnn_b200: activations left the range of precision={target.precision!r} storage "
                                     "(encoder hidden layer); run this checkpoint with precision='tf32' or 'fp32'")

    def _begin_graph_index(self, edge_index, batch, n):
        """Returns an object with .finish() -> GraphIndex (cached index when cache_index is on).

        `cache_index=True` reuses the CSR while the caller passes THE SAME tensor objects, unmodified: the key is the
        identity of `edge_index` / `batch` (held through weak references, so a recycled id or a recycled allocator
        address cannot alias a dead tensor) plus their version counters.  A new tensor with equal contents rebuilds."""
        if self.cache_index:
            import weakref
            c = self._index_cache
            if (c is not None and c["ei"]() is edge_index and c["ei_v"] == edge_index._version and c["n"] == n
                    and ((batch is None and c["b"] is None) or
                         (batch is not None and c["b"] is not None and c["b"]() is batch and c["b_v"] == batch._version))):
                cached = c["idx"]
                return type("Cached", (), {"finish": staticmethod(lambda: cached)})
            pending = engine.begin_graph_index(edge_index, batch, n)
            outer = self
            entry = {"ei": weakref.ref(edge_index), "ei_v": edge_index._version, "n": n,
                     "b": None if batch is None else weakref.ref(batch), "b_v": None if batch is None else batch._version}

            class _Fill:
                @staticmethod
                def finish():
                    idx = pending.finish()
                    outer._index_cache = dict(entry, idx=idx)
                    return idx
            return _Fill
        return engine.begin_graph_index(edge_index, batch, n)

    def _forward_cuda_eagnn(self, x, edge_index, edge_attr, batch, node_level=False, width=512):
        """EA-GNN / "CustomGNN" path (reference :326-336, :375-387, GraphNetBlock :528-566).  `width` 128: a
        hidden_channels = 128 model on the 128-wide kernels."""
        packs = self._packed(width)
        prec, cg = self.precision, self.cta_group
        x = x.detach().to(torch.float32).contiguous()
        if not edge_attr.is_cuda:
            raise RuntimeError("buckgnn_b200: `edge_attr` must be a CUDA tensor")
        edge_attr = edge_attr.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        # GraphNetBlock aggregates on row = edge_index[0] (:553,561) -> CSR keyed by row 0
        pending = engine.begin_graph_index(edge_index, batch, n, key_row=0)
        cur = Activation(n, width, prec, x.device)
        flag = self._new_nonfinite_flag(x.device)
        engine.encoder_forward(x, packs["enc"], packs["enc_w3"], prec, cur, cg, nonfinite=flag)  # :323
        idx = pending.finish()
        ne = idx.n_edges
        ex = engine.edge_extras(idx, prec)
        e = Activation(max(ne, 1), width, prec, x.device)
        if ne > 0:                                   # edge_encoder on edge_attr in CSR order (:327, :376)
            engine.encoder_forward(edge_attr, packs["edge_enc"], packs["edge_enc_w3"], prec, e, cg,
                                   row_gather=idx.perm[:ne], nonfinite=flag)
        buf = engine.GNBlockBuffers(n, ne, prec, x.device, width)
        L = self.num_layers
        for i, w in enumerate(packs["gn"]):
            cur, e_next = engine.gnblock_layer(cur, e, buf, idx, ex, w, skip=(0 < i < L - 1),
                                               need_edges_out=(i < L - 1), cta_group=cg)
            if e_next is not None:
                e = e_next
        if node_level:
            return engine.node_head(cur, n, packs["node_head"], self.output_dim, cg)
        pre = packs["pool_mlp"] if self.pooling_layer in ("mlp", "mlp_no_super") else None
        pred, _ = engine.pool_head(cur, idx, packs["dec"], self.output_dim, pooling=self.pooling_layer, pre=pre,
                                   nonfinite=flag)
        return pred

    def _forward_cuda(self, x, edge_index, batch, node_level=False, width=512):
        """`width` 128: a hidden_channels = 128 model on the 128-wide kernels (bg_gemm128, bg_pool_head128)."""
        packs = self._packed(width)
        prec, cg = self.precision, self.cta_group
        x = x.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        pending = self._begin_graph_index(edge_index, batch, n)       # K1 enqueued, result read-back in flight
        cur = Activation(n, width, prec, x.device)
        layers = packs["layers"]
        folded = packs["layer0_folded"]
        flag = self._new_nonfinite_flag(x.device)
        if folded is not None:
            h = engine.encoder_hidden(x, packs["enc"], prec, nonfinite=flag)          # reference :323, first two Linears
        else:
            engine.encoder_forward(x, packs["enc"], packs["enc_w3"], prec, cur, cg, nonfinite=flag)      # reference :323
        idx = pending.finish()                                        # host sync hidden behind the encoder
        blocks = None
        if layers:
            nxt = Activation(n, width, prec, x.device)
            agg = Activation(n, width, prec, x.device)
            aggr = self._sage_layers()[0][0].aggr
            L = len(layers)
            for i, layer in enumerate(layers):                                            # reference :445-458
                if i == 0 and folded is not None:                     # encoder's last Linear folded into layer 0
                    engine.sage_layer0_folded(h, nxt, idx, folded, aggr=aggr, normalize=True, relu=True,
                                              cta_group=cg)
                else:
                    residual = 0 < i < L - 1
                    # the last layer's rows are only read by the pooling layer (:515), which is linear in them:
                    # its epilogue sums them per 32-row block instead of storing them (16-bit modes)
                    if (i == L - 1 and not node_level and self.fuse_pool
                            and engine.can_fuse_pool(prec, True, residual)):
                        blocks = engine.new_pool_blocks(idx, x.device, width)
                    engine.sage_layer(cur, agg, nxt, idx, layer, aggr=aggr, normalize=True, relu=True,
                                      residual=residual, cta_group=cg, pool_blocks=blocks,
                                      fuse_aggregate=self.fuse_aggregate)
                cur, nxt = nxt, cur
        if node_level:
            return engine.node_head(cur, n, packs["node_head"], self.output_dim, cg)     # reference :518-524
        pre = packs["pool_mlp"] if self.pooling_layer in ("mlp", "mlp_no_super") else None
        pred, _ = engine.pool_head(cur, idx, packs["dec"], self.output_dim, pooling=self.pooling_layer,
                                   pre=pre, nonfinite=flag, blocks=blocks)                 # reference :515-516
        return pred

    # ------------------------------------------------------------------ SAGPooling variants (SURVEY.md section 8 row f4)
    def _tail(self, cur, idx, packs, node_level, cg):
        if node_level:
            return engine.node_head(cur, idx.n_nodes, packs["node_head"], self.output_dim, cg)
        pre = packs["pool_mlp"] if self.pooling_layer in ("mlp", "mlp_no_super") else None
        pred, _ = engine.pool_head(cur, idx, packs["dec"], self.output_dim, pooling=self.pooling_layer, pre=pre)
        return pred

    def _forward_cuda_sag(self, x, edge_index, edge_attr, batch, node_level=False):
        """`GraphSAGE_SAG` (reference :190-217, :493-511): num_layers // 2 SAGE('add') layers, SAGPooling(0.5),
        the remaining layers on the pooled graph, every layer after the first with a skip."""
        packs = self._packed()
        prec, cg = self.precision, self.cta_group
        x = x.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        pending = engine.begin_graph_index(edge_index, batch, n)
        layers = packs["layers"]
        n_before = len(self.sage_layers_1)
        folded = packs["layer0_folded"] if n_before > 0 else None
        cur = Activation(n, 512, prec, x.device)
        if folded is not None:
            h = engine.encoder_hidden(x, packs["enc"], prec)
        else:
            engine.encoder_forward(x, packs["enc"], packs["enc_w3"], prec, cur, cg)
        idx = pending.finish()
        if n_before > 0:
            nxt = Activation(n, 512, prec, x.device)
            agg = Activation(n, 512, prec, x.device)
            for i in range(n_before):
                if i == 0 and folded is not None:
                    engine.sage_layer0_folded(h, nxt, idx, folded, aggr="add", normalize=True, relu=True, cta_group=cg)
                else:
                    engine.sage_layer(cur, agg, nxt, idx, layers[i], aggr="add", normalize=True, relu=True,
                                      residual=(i > 0), cta_group=cg)
                cur, nxt = nxt, cur
            del nxt, agg
        pooled = engine.sag_pool(cur, idx, idx.graph_ptr, idx.n_graphs, edge_index, packs["sag_pool"], sign=self._sag_sign)
        self.last_pool = engine.pool_summary(pooled)   # perm / score / edge_index / batch of the last pooling, without its feature rows
        idx2 = engine.build_graph_index(pooled.edge_index, pooled.batch, pooled.n_nodes)
        cur = pooled.x
        n2 = pooled.n_nodes
        nxt = Activation(n2, 512, prec, x.device)
        agg = Activation(n2, 512, prec, x.device)
        for layer in layers[n_before:]:
            engine.sage_layer(cur, agg, nxt, idx2, layer, aggr="add", normalize=True, relu=True, residual=True,
                              cta_group=cg)
            cur, nxt = nxt, cur
        return self._tail(cur, idx2, packs, node_level, cg), pooled.batch

    def _forward_cuda_eagnn_sag(self, x, edge_index, edge_attr, batch, node_level=False):
        """`EAGNN_SAG` (reference :219-244, :354-373): GraphNetBlocks around a SAGPooling; the pooled edge features are
        the rows of the kept edges."""
        packs = self._packed()
        prec, cg = self.precision, self.cta_group
        x = x.detach().to(torch.float32).contiguous()
        if not edge_attr.is_cuda:
            raise RuntimeError("buckgnn_b200: `edge_attr` must be a CUDA tensor")
        edge_attr = edge_attr.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        pending = engine.begin_graph_index(edge_index, batch, n, key_row=0)       # GraphNetBlock direction (:553, :561)
        pending_t = engine.begin_graph_index(edge_index, None, n, key_row=1)      # SAGEConv direction of the score GNN
        cur = Activation(n, 512, prec, x.device)
        engine.encoder_forward(x, packs["enc"], packs["enc_w3"], prec, cur, cg)
        idx = pending.finish()
        idx_t = pending_t.finish()
        ne = idx.n_edges
        e = Activation(max(ne, 1), 512, prec, x.device)
        if ne > 0:
            engine.encoder_forward(edge_attr, packs["edge_enc"], packs["edge_enc_w3"], prec, e, cg,
                                   row_gather=idx.perm[:ne])
        if packs["gn1"]:
            ex = engine.edge_extras(idx, prec)
            buf = engine.GNBlockBuffers(n, ne, prec, x.device)
            for i, w in enumerate(packs["gn1"]):
                cur, e_next = engine.gnblock_layer(cur, e, buf, idx, ex, w, skip=(i > 0), need_edges_out=True, cta_group=cg)
                e = e_next
        pooled = engine.sag_pool(cur, idx_t, idx.graph_ptr, idx.n_graphs, edge_index, packs["sag_pool"],
                                 sign=self._sag_sign, want_kept_edges=True)
        self.last_pool = engine.pool_summary(pooled)   # perm / score / edge_index / batch of the last pooling, without its feature rows
        idx2 = engine.build_graph_index(pooled.edge_index, pooled.batch, pooled.n_nodes, key_row=0)
        e = engine.regather_edge_rows(e, idx, idx2, pooled.kept_edge)
        cur = pooled.x
        n2, ne2 = pooled.n_nodes, idx2.n_edges
        ex2 = engine.edge_extras(idx2, prec)
        buf2 = engine.GNBlockBuffers(n2, ne2, prec, x.device)
        last = len(packs["gn2"]) - 1
        for i, w in enumerate(packs["gn2"]):
            cur, e_next = engine.gnblock_layer(cur, e, buf2, idx2, ex2, w, skip=True, need_edges_out=(i < last), cta_group=cg)
            if e_next is not None:
                e = e_next
        return self._tail(cur, idx2, packs, node_level, cg), pooled.batch
