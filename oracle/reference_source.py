"""Runs the reference's OWN `Models/BuckGNN.py`, unmodified, on the CPU.  TEST INFRASTRUCTURE ONLY.

The reference file imports two third-party packages that are not installable here
(`torch_geometric`, `torch_scatter`; `Models/BuckGNN.py:3-6`).  `install_shims()` registers
minimal stand-ins for exactly the names that file imports -- `SAGEConv`, `SAGPooling`,
`global_{mean,max,add}_pool`, `scatter_add`, `scatter_mean` -- with the constructor / call
signatures PyG and torch_scatter publish, backed by the operator functions of
`oracle/buckgnn_oracle.py`.  `load_reference()` then executes the reference source file where it
lies (`Models/BuckGNN.py` of a checkout of the reference project; nothing is copied), so the reference's real
constructor, layer loops, skip rules, pooling selection, `.squeeze()` and error branches run as
written.  What stays restated is only the arithmetic inside the two third-party packages.

Used by `tests/test_reference_source.py` (the reference re-run against its stored outputs) and by
`tests/golden/make_golden.py` / `make_reference_cases.py` (the committed fixtures are outputs of the reference file).
The reference project is not part of this repository: set BUCKGNN_REFERENCE_DIR to a checkout of it.
Without one, callers must check `reference_available()`.
"""
from __future__ import annotations

import hashlib
import importlib.util
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import buckgnn_oracle as O

REFERENCE_DIR = os.environ.get("BUCKGNN_REFERENCE_DIR", "")
REFERENCE_FILE = os.path.join(REFERENCE_DIR, "Models", "BuckGNN.py") if REFERENCE_DIR else ""
SKIP_REASON = "needs a checkout of the reference project (github.com/omerkurt-okt/buck-gnn): set BUCKGNN_REFERENCE_DIR"


def reference_available(path: str = REFERENCE_FILE) -> bool:
    return bool(path) and os.path.isfile(path)


def reference_sha256(path: str = REFERENCE_FILE) -> str:
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


# ----------------------------------------------------------------------------- torch_scatter stand-ins
def _scatter(src, index, dim, dim_size, reduce):
    """torch_scatter / torch_geometric.utils.scatter for a 1-D `index` along `dim`."""
    dim = dim if dim >= 0 else src.dim() + dim
    moved = src.movedim(dim, 0)
    if dim_size is None:
        dim_size = int(index.max()) + 1 if index.numel() > 0 else 0
    fn = {"sum": O.scatter_sum, "mean": O.scatter_mean, "max": O.scatter_max}[reduce]
    return fn(moved, index, dim_size).movedim(0, dim)


def scatter_add(src, index, dim=-1, out=None, dim_size=None):
    assert out is None
    return _scatter(src, index, dim, dim_size, "sum")


def scatter_mean(src, index, dim=-1, out=None, dim_size=None):
    assert out is None
    return _scatter(src, index, dim, dim_size, "mean")


# ----------------------------------------------------------------------------- torch_geometric.nn stand-ins
def _global_pool(x, batch, size, reduce):
    """PyG `global_*_pool`: dim = -2 (node dimension) unless x is 1-D; `batch=None` reduces over all nodes and
    keeps the dimension for inputs of at most two dimensions."""
    dim = -1 if x.dim() == 1 else -2
    if batch is None:
        keep = x.dim() <= 2
        if reduce == "mean":
            return x.mean(dim=dim, keepdim=keep)
        if reduce == "sum":
            return x.sum(dim=dim, keepdim=keep)
        return x.max(dim=dim, keepdim=keep)[0]
    return _scatter(x, batch, dim, size, reduce)


def global_mean_pool(x, batch, size=None):
    return _global_pool(x, batch, size, "mean")


def global_add_pool(x, batch, size=None):
    return _global_pool(x, batch, size, "sum")


def global_max_pool(x, batch, size=None):
    return _global_pool(x, batch, size, "max")


class SAGEConv(nn.Module):
    """PyG `SAGEConv(in_channels, out_channels, aggr='mean', normalize=False, root_weight=True, project=False,
    bias=True)`: parameters `lin_l.{weight,bias}`, `lin_r.weight`."""

    def __init__(self, in_channels, out_channels, aggr="mean", normalize=False, root_weight=True, project=False,
                 bias=True, **kwargs):
        super().__init__()
        assert root_weight and not project and not kwargs, "not used by the reference"
        self.in_channels, self.out_channels = in_channels, out_channels
        self.aggr, self.normalize = aggr, normalize
        self.lin_l = nn.Linear(in_channels, out_channels, bias=bias)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, edge_index, size=None):
        out = self.lin_l(O.aggregate(x, edge_index, self.aggr)) + self.lin_r(x)
        if self.normalize:
            out = F.normalize(out, p=2.0, dim=-1)
        return out


class SAGPooling(nn.Module):
    """PyG `SAGPooling(in_channels, ratio=0.5, GNN=GraphConv, min_score=None, multiplier=1.0,
    nonlinearity='tanh', **kwargs)` with `self.gnn = GNN(in_channels, 1, **kwargs)` (the PyG < 2.4 layout the
    reference's checkpoints have)."""

    def __init__(self, in_channels, ratio=0.5, GNN=None, min_score=None, multiplier=1.0, nonlinearity="tanh", **kwargs):
        super().__init__()
        assert GNN is not None and min_score is None and multiplier == 1.0 and nonlinearity == "tanh"
        self.in_channels, self.ratio = in_channels, ratio
        self.gnn = GNN(in_channels, 1, **kwargs)

    def forward(self, x, edge_index, edge_attr=None, batch=None, attn=None):
        if batch is None:
            batch = edge_index.new_zeros(x.size(0))
        attn = x if attn is None else attn
        attn = attn.unsqueeze(-1) if attn.dim() == 1 else attn
        score = torch.tanh(self.gnn(attn, edge_index).view(-1))
        perm = O.topk(score, self.ratio, batch)
        x = x[perm] * score[perm].view(-1, 1)
        batch = batch[perm]
        edge_index, edge_attr = O.filter_adj(edge_index, edge_attr, perm, num_nodes=score.size(0))
        return x, edge_index, edge_attr, batch, perm, score[perm]


_SHIM_NAMES = ("torch_geometric", "torch_geometric.nn", "torch_scatter")


def install_shims() -> dict:
    """Registers the stand-in packages in sys.modules (refuses to shadow a real install); returns what was there."""
    saved = {k: sys.modules.get(k) for k in _SHIM_NAMES}
    for k, v in saved.items():
        if v is not None and not getattr(v, "__buckgnn_shim__", False):
            raise RuntimeError(f"{k} is really installed: import the reference directly instead of shimming it")
    tg = types.ModuleType("torch_geometric")
    tgnn = types.ModuleType("torch_geometric.nn")
    ts = types.ModuleType("torch_scatter")
    for m in (tg, tgnn, ts):
        m.__buckgnn_shim__ = True
    for name in ("SAGEConv", "SAGPooling", "global_mean_pool", "global_max_pool", "global_add_pool"):
        setattr(tgnn, name, globals()[name])
    tg.nn = tgnn
    ts.scatter_add, ts.scatter_mean = scatter_add, scatter_mean
    sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": tgnn, "torch_scatter": ts})
    return saved


def remove_shims(saved: dict) -> None:
    for k in _SHIM_NAMES:
        if saved.get(k) is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = saved[k]


_CACHE = {}


def load_reference(path: str = REFERENCE_FILE):
    """Executes the reference's model file (unmodified, read where it lies) under the shims and returns the module:
    `.BuckGNN`, `.GraphNetBlock`, `.MLPPooling`, `.HybridPooling`."""
    if path in _CACHE:
        return _CACHE[path]
    if not reference_available(path):
        raise FileNotFoundError(path)
    saved = install_shims()
    try:
        spec = importlib.util.spec_from_file_location("_reference_Models_BuckGNN", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        remove_shims(saved)
    mod.__reference_sha256__ = reference_sha256(path)
    _CACHE[path] = mod
    return mod
