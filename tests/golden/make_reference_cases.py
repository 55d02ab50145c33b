"""Generates tests/golden/reference_cases.json.gz: what the reference's own `Models/BuckGNN.py` returns for every case of
tests/test_reference_source.py, so that those comparisons run without a checkout of the reference project.

    BUCKGNN_REFERENCE_DIR=<checkout of the reference project> python tests/golden/make_reference_cases.py
    python tests/golden/make_reference_cases.py --without-reference

The committed file was written with --without-reference from a tree whose oracle/, Models/, buckgnn_b200/ and
tests/ are identical to commit 0c3dd9f.  At that commit every case below was run through the reference file (sha256
in tests/golden/oracle_golden.json) and matched what --without-reference stores for it, to the tolerances of
tests/test_reference_source.py: the oracle's outputs, the product's constructor for the state_dict contract (the
side the reference's constructor was compared with), and for the single case where the oracle does not reproduce a
failure of the reference (REFERENCE_FAILURES below), the exception the reference raised.  Where a
checkout is present, the tests re-run the reference and check it against this file as well.

A case is built by `run_case(kind, cls, **params)` with `cls` the reference's `BuckGNN` or a class with the same
constructor (the oracle, the product): seeded weights, non-trivial BN statistics, a seeded synthetic batch.  It
returns a flat dict of tensors / lists / strings / None.  Gradients are stored as their norms plus a seeded sample of
64 entries per parameter; the file is gzip-compressed JSON, tensors as {"dtype", "shape", "data"}.
"""
import gzip
import itertools
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch

from buckgnn_b200.synth import make_batch
from oracle import buckgnn_oracle as O
from oracle import reference_source as RS

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "reference_cases.json.gz")

WORKING = ["GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr",
           "GraphSage_addAggr_Shared", "EA_GNN", "EA_GNN_Shared", "GraphSAGE_SAG", "EAGNN_SAG", "GraphSAGE_MLP"]
BROKEN = ["GraphSage_MLP", "GraphSage_addAggr_woBatchNorm", "GraphSage_sumAggr_woBatchNorm"]
POOLINGS = ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super"]
HEADS = [("static_disp", False, False, 2), ("static_disp", True, False, 3), ("static_disp", False, True, 4),
         ("static_disp", True, True, 6), ("static_stress", False, False, 3), ("mode_shape", False, False, 3),
         ("mode_shape", False, True, 6)]
GRAD_SAMPLE = 64


def seeded(cls, seed=0, **cfg):
    """Same constructor order -> same RNG stream: the reference and the oracle get identical parameters."""
    base = dict(num_node_features=16, num_edge_features=5, hidden_channels=256, num_layers=4,
                pooling_layer="mean", model_name="GraphSage_meanAggr", dropout_rate=0.0)
    base.update(cfg)
    torch.manual_seed(seed)
    m = cls(**base)
    O.randomize_bn_stats(m, realistic=True)
    return m


def state_checksum(m):
    return sum((i + 1) * float(t.double().sum()) for i, t in enumerate(m.state_dict().values()))


def _forward(m, b, with_batch=True):
    with torch.no_grad():
        pred, bout = m.eval()(b.x, b.edge_index, b.edge_attr, b.batch if with_batch else None)
    return {"state_checksum": state_checksum(m), "pred": pred, "batch": bout}


def _ctor(m):
    sd = m.state_dict()
    return {"keys": list(sd), "shapes": [list(v.shape) for v in sd.values()], "dtypes": [str(v.dtype) for v in sd.values()],
            "parameters": [n for n, _ in m.named_parameters()]}


def run_case(kind, cls, **p):
    if kind == "forward":                  # every working model_name at two widths
        stiff = p["name"] in ("EA_GNN", "EA_GNN_Shared", "EAGNN_SAG")
        b = make_batch(num_graphs=3, nx=6, ny=5, stiffened=stiff)
        m = seeded(cls, model_name=p["name"], hidden_channels=p["hidden"])
        out = _forward(m, b)
        if "SAG" not in p["name"].replace("GraphSAGE_MLP", ""):
            with torch.no_grad():                                  # Models/BuckGNN.py:516 returns the input object
                out["batch_is_input"] = m(b.x, b.edge_index, b.edge_attr, b.batch)[1] is b.batch
        return out
    if kind == "pooling":                  # every pooling layer
        return _forward(seeded(cls, model_name=p["name"], pooling_layer=p["pooling"], num_layers=3),
                        make_batch(num_graphs=3, nx=5, ny=4, stiffened=p["name"] == "EA_GNN"))
    if kind == "batch_none":               # one graph, batch=None
        m, b = seeded(cls, pooling_layer=p["pooling"], num_layers=2), make_batch(num_graphs=1, nx=5, ny=4)
        try:
            return _forward(m, b, with_batch=False)
        except Exception as e:              # noqa: BLE001 - the exception type is the stored outcome
            return {"raises": type(e).__name__}
    if kind == "heads":                    # node-level prediction types
        return _forward(seeded(cls, prediction_type=p["ptype"], use_z_coord=p["z"], use_rotations=p["rot"],
                               pooling_layer=p["pooling"], num_layers=2), make_batch(num_graphs=2, nx=5, ny=4))
    if kind == "one_graph":                # one graph WITH its batch vector: .squeeze() to 0-dim
        return _forward(seeded(cls, num_layers=2), make_batch(num_graphs=1, nx=5, ny=4))
    if kind == "ctor":                     # state_dict contract for every (pooling, prediction_type)
        out = {}
        for pooling, ptype in itertools.product(["mean", "supernode_with_pooling"], ["buckling", "static_stress"]):
            m = cls(num_node_features=16, num_edge_features=5, hidden_channels=p["hidden"], num_layers=3,
                    pooling_layer=pooling, prediction_type=ptype, model_name=p["name"])
            out.update({f"{pooling}.{ptype}.{k}": v for k, v in _ctor(m).items()})
        return out
    if kind == "broken":                   # model names whose forward fails in the reference: the ctor still builds
        return _ctor(cls(16, 5, 256, 2, "mean", model_name=p["name"]))
    if kind == "train":                    # one training step: loss, gradients, BN buffers after it
        m = seeded(cls, model_name=p["name"], num_layers=3, hidden_channels=128).train()
        b = make_batch(num_graphs=3, nx=5, ny=4, stiffened=p["name"] == "EA_GNN")
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
        loss = torch.nn.functional.mse_loss(pred, torch.tensor([0.5, -0.25, 1.0]))
        loss.backward()
        out = {"state_checksum": state_checksum(m), "loss": loss.detach(),
               "no_grad": sorted(k for k, q in m.named_parameters() if q.grad is None)}
        for k, q in m.named_parameters():
            if q.grad is not None:
                g = q.grad.reshape(-1)
                idx = torch.randperm(g.numel(), generator=torch.Generator().manual_seed(0))[:GRAD_SAMPLE].sort().values
                out[f"grad_norm.{k}"] = g.double().norm()
                out[f"grad_index.{k}"] = idx
                out[f"grad.{k}"] = g[idx]
        out.update({f"buf.{k}": v.detach().clone() for k, v in m.named_buffers()})
        return out
    if kind == "errors":                   # the reference's failure branches: the exception type of each
        b = make_batch(num_graphs=2, nx=4, ny=4)

        def outcome(build, forward=True):
            try:
                m = build()
                if forward:
                    with torch.no_grad():
                        m.eval()(b.x, b.edge_index, b.edge_attr, b.batch)
                return "none"
            except Exception as e:          # noqa: BLE001 - the exception type is the stored outcome
                return type(e).__name__
        out = {"unknown_pooling": outcome(lambda: cls(16, 5, 256, 2, "nope", model_name="GraphSage_meanAggr")),
               "hybrid_pooling": outcome(lambda: cls(16, 5, 256, 2, "hybrid", model_name="GraphSage_meanAggr")),
               "unknown_prediction_type": outcome(lambda: cls(16, 5, 256, 2, "mean", prediction_type="nope"), forward=False),
               "hidden_200": outcome(lambda: cls(16, 5, 200, 2, "mean", model_name="GraphSage_meanAggr"))}
        out.update({f"broken.{n}": outcome(lambda n=n: cls(16, 5, 256, 2, "mean", model_name=n)) for n in BROKEN})
        return out
    if kind == "dropout":                  # dropout follows torch's RNG stream
        m = seeded(cls, num_layers=3, hidden_channels=128, dropout_rate=0.3).train()
        b = make_batch(num_graphs=2, nx=5, ny=4)
        torch.manual_seed(123)
        return {"pred": m(b.x, b.edge_index, b.edge_attr, b.batch)[0].detach()}
    raise ValueError(kind)


def cases():
    """(key, kind, params) of every stored case."""
    out = [(f"forward/{n}/{h}", "forward", dict(name=n, hidden=h)) for n in WORKING for h in (128, 256)]
    out += [(f"pooling/{n}/{q}", "pooling", dict(name=n, pooling=q))
            for n in ("GraphSage_meanAggr", "EA_GNN", "GraphSAGE_SAG") for q in POOLINGS]
    out += [(f"batch_none/{q}", "batch_none", dict(pooling=q)) for q in POOLINGS]
    out += [(f"heads/{t}/{z}/{r}/{q}", "heads", dict(ptype=t, z=z, rot=r, pooling=q))
            for t, z, r, _ in HEADS for q in ("mean", "supernode_only")]
    out += [("one_graph", "one_graph", {})]
    out += [(f"ctor/{n}/{h}", "ctor", dict(name=n, hidden=h)) for n in WORKING + BROKEN[:2] for h in (128, 512)]
    out += [(f"broken/{n}", "broken", dict(name=n)) for n in BROKEN]
    out += [(f"train/{n}", "train", dict(name=n)) for n in ("GraphSage_meanAggr", "GraphSage_maxAggr", "EA_GNN", "GraphSAGE_SAG")]
    out += [("dropout", "dropout", {})]
    out += [("errors", "errors", {})]
    return out


# What the reference raised where the oracle deliberately does not fail (a NameError entry also matches its
# subclass UnboundLocalError).  --without-reference stores these instead of the oracle's outcome.
REFERENCE_FAILURES = {
    # cat of a [1,1,H] pooled tensor with a [1,H] super-node row (Models/BuckGNN.py:285-292)
    "batch_none/supernode_with_pooling": {"raises": "RuntimeError"},
    "errors": {"unknown_pooling": "ValueError",
               "hybrid_pooling": "AttributeError",          # hybrid_pooling is commented out (:188)
               "unknown_prediction_type": "NameError",      # output_dim never bound (:19-38)
               "hidden_200": "AttributeError",              # 129..255: no encoder is built (:41,67)
               # module lists only built under OTHER names (:404,417,472)
               **{f"broken.{n}": "AttributeError" for n in BROKEN}},
}


def encode(v):
    if isinstance(v, torch.Tensor):
        return {"dtype": str(v.dtype).replace("torch.", ""), "shape": list(v.shape), "data": v.reshape(-1).tolist()}
    return v


def decode(v):
    if isinstance(v, dict) and set(v) == {"dtype", "shape", "data"}:
        return torch.tensor(v["data"], dtype=getattr(torch, v["dtype"])).reshape(v["shape"])
    return v


def load():
    with gzip.open(PATH, "rt") as f:
        data = json.load(f)
    return {key: {k: decode(v) for k, v in case.items()} for key, case in data["cases"].items()}


def main():
    without = "--without-reference" in sys.argv
    if not without and not RS.reference_available():
        raise SystemExit("make_reference_cases.py runs the reference's own Models/BuckGNN.py: " + RS.SKIP_REASON)
    from buckgnn_b200.model import BuckGNN
    data = {"source": "without-reference" if without else "reference", "cases": {}}
    for key, kind, params in cases():
        if not without:
            cls = RS.load_reference().BuckGNN
        else:
            cls = BuckGNN if kind in ("ctor", "broken") else O.OracleBuckGNN
        if without and key in REFERENCE_FAILURES:
            case = REFERENCE_FAILURES[key]
        else:
            case = run_case(kind, cls, **params)
        data["cases"][key] = {k: encode(v) for k, v in case.items()}
    with gzip.GzipFile(PATH, "wb", mtime=0) as f:
        f.write(json.dumps(data, separators=(",", ":")).encode())
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
