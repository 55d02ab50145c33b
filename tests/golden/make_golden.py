"""Generates tests/golden/oracle_golden.json by RUNNING THE REFERENCE'S OWN FILE.

    BUCKGNN_REFERENCE_DIR=<checkout of the reference project> python tests/golden/make_golden.py

The model that produces every stored number is `BuckGNN` from the reference's `Models/BuckGNN.py`,
executed unmodified through `oracle/reference_source.py` (its two third-party imports, torch_geometric
and torch_scatter -- not installable here -- are shimmed with stand-ins of the same signatures, backed by
the restated operators of oracle/buckgnn_oracle.py).  The file records the sha256 of the reference source
it ran.  Inputs are regenerated from seeds (buckgnn_b200.synth, torch.manual_seed); outputs are stored.
Without a reference checkout, tests read the committed JSON; `seeded_model` there builds the
oracle twin with the same seed as a WEIGHT CONTAINER (its state_dict checksum is checked against the file).
"""
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

FORWARD_CASES = [  # name, model cfg overrides, batch kwargs
    ("sage_mean_6x512", dict(model_name="GraphSage_meanAggr"), dict(num_graphs=3, nx=9, ny=7)),
    ("sage_sum_4x512", dict(model_name="GraphSage_sumAggr", num_layers=4), dict(num_graphs=2, nx=8, ny=6)),
    ("sage_max_4x512", dict(model_name="GraphSage_maxAggr", num_layers=4), dict(num_graphs=2, nx=8, ny=6)),
    ("sage_add_shared_4x512", dict(model_name="GraphSage_addAggr_Shared", num_layers=4), dict(num_graphs=2, nx=8, ny=6)),
    ("eagnn_3x512_stiffened", dict(model_name="EA_GNN", num_layers=3), dict(num_graphs=2, nx=7, ny=6, stiffened=True)),
    ("default_mlp", dict(model_name="GraphSAGE_MLP"), dict(num_graphs=3, nx=6, ny=5)),
    # TRAIN_FINAL.py:55,71 and the constructor default: hidden_channels=128 (2-layer encoder / decoder, :41-65)
    ("sage_mean_6x128", dict(model_name="GraphSage_meanAggr", hidden_channels=128), dict(num_graphs=3, nx=9, ny=7)),
    ("sage_add_4x128_mlp_pool", dict(model_name="GraphSage_addAggr", hidden_channels=128, num_layers=4, pooling_layer="mlp"),
     dict(num_graphs=2, nx=8, ny=6)),
    ("eagnn_3x128_stiffened", dict(model_name="EA_GNN", hidden_channels=128, num_layers=3), dict(num_graphs=2, nx=7, ny=6, stiffened=True)),
    ("sage_mean_4x256", dict(model_name="GraphSage_meanAggr", hidden_channels=256, num_layers=4), dict(num_graphs=2, nx=8, ny=6)),
    # configs[4]'s model on its meshes: stiffened plates with virtual edges + super node
    ("sage_mean_6x512_stiffened_virtual", dict(model_name="GraphSage_meanAggr"), dict(num_graphs=3, nx=9, ny=8, stiffened=True)),
    ("sage_mean_6x512_no_super_virtual", dict(model_name="GraphSage_meanAggr"),
     dict(num_graphs=2, nx=9, ny=8, stiffened=True, super_node=False, virtual_edges=True)),
    ("sage_mean_supernode_only", dict(model_name="GraphSage_meanAggr", num_layers=3, pooling_layer="supernode_only"),
     dict(num_graphs=3, nx=6, ny=5)),
    # SAGPooling variants: the top-k is discrete, so these cases are chosen (and checked below) to have a clear
    # score gap at every graph's keep/drop threshold -- tf32 rounding cannot flip the selection
    ("sage_sag_6x512", dict(model_name="GraphSAGE_SAG"), dict(num_graphs=3, nx=9, ny=7)),
    ("eagnn_sag_4x512_stiffened", dict(model_name="EAGNN_SAG", num_layers=4), dict(num_graphs=2, nx=7, ny=6, stiffened=True)),
]
MIN_TOPK_GAP = 1e-3


def model_cfg(**over):
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=512, num_layers=6,
               pooling_layer="mean", model_name="GraphSage_meanAggr")
    cfg.update(over)
    return cfg


def seeded_model(cfg, reference: bool):
    """Seeded weights + non-trivial BN statistics.  reference=True: the class from the reference's own file;
    False: the oracle twin (same constructor order -> same RNG stream -> identical state_dict)."""
    torch.manual_seed(0)
    m = (RS.load_reference().BuckGNN if reference else O.OracleBuckGNN)(**cfg)
    O.randomize_bn_stats(m, realistic=True)
    return m


def seeded_oracle(cfg):
    return seeded_model(cfg, reference=False)


def state_checksum(m):
    """Order-sensitive fp64 checksum of the seeded parameters and buffers (detects RNG drift)."""
    s = 0.0
    for i, (_, t) in enumerate(m.state_dict().items()):
        s += (i + 1) * float(t.double().sum())
    return s


def kat():
    """The 5-node / 2-graph case of tests/test_oracle.py: an isolated node and a hub."""
    x = torch.arange(10, dtype=torch.float32).view(5, 2) / 4 - 1
    ei = torch.tensor([[0, 1, 3, 3, 0, 1], [2, 2, 2, 4, 1, 0]])
    batch = torch.tensor([0, 0, 0, 1, 1])
    return x, ei, batch


def sag_kat():
    """Hand-checkable SAGPooling index work: 2 graphs (5 + 3 nodes), ties inside both.
    graph 0 keeps ceil(2.5) = 3 of scores [.3, .9, .9, -.2, .5] -> nodes 1, 2 (tie: lower id first), 4;
    graph 1 keeps ceil(1.5) = 2 of [.1, .7, .7] -> nodes 6, 7."""
    score = torch.tensor([0.3, 0.9, 0.9, -0.2, 0.5, 0.1, 0.7, 0.7])
    batch = torch.tensor([0, 0, 0, 0, 0, 1, 1, 1])
    ei = torch.tensor([[0, 1, 2, 4, 1, 4, 5, 6, 7, 6], [1, 2, 1, 2, 4, 3, 6, 7, 6, 5]])
    return score, batch, ei


def topk_gaps(m, b):
    """Per graph: score gap between the last kept and the first dropped node of the oracle's SAGPooling."""
    cap = {}

    def hook(mod, inp, out):
        cap["score"] = torch.tanh(mod.gnn(inp[0], inp[1]).view(-1))
        cap["batch"] = inp[3]
    h = m.pool.register_forward_hook(hook)
    with torch.no_grad():
        m(b.x, b.edge_index, b.edge_attr, b.batch)
    h.remove()
    gaps = []
    for g in range(int(cap["batch"].max()) + 1):
        sg = cap["score"][cap["batch"] == g].sort(descending=True).values
        k = -(-len(sg) // 2)
        gaps.append(float(sg[k - 1] - sg[k]) if k < len(sg) else float("inf"))
    return gaps


def main():
    if not RS.reference_available():
        raise SystemExit("make_golden.py runs the reference's own Models/BuckGNN.py: " + RS.SKIP_REASON)
    out = {"generated_from": os.path.relpath(RS.REFERENCE_FILE, RS.REFERENCE_DIR), "reference_sha256": RS.reference_sha256(),
           "generator": "tests/golden/make_golden.py via oracle/reference_source.py (torch_geometric / torch_scatter shimmed)",
           "forward": {}, "operators": {}, "training": {}}
    for name, over, bkw in FORWARD_CASES:
        cfg = model_cfg(**over)
        m = seeded_model(cfg, reference=True).eval()
        b = make_batch(**bkw)
        with torch.no_grad():
            pred, bout = m(b.x, b.edge_index, b.edge_attr, b.batch)
        out["forward"][name] = {"cfg": cfg, "batch": bkw, "nodes": b.num_nodes, "edges": b.num_edges,
                                "state_checksum": state_checksum(m), "pred": pred.double().reshape(-1).tolist()}
        if hasattr(m, "pool"):
            gaps = topk_gaps(m, b)
            assert min(gaps) > MIN_TOPK_GAP, (name, gaps)
            out["forward"][name].update(pooled_nodes=int(bout.shape[0]), min_topk_gap=min(gaps))
    x, ei, batch = kat()
    ops = out["operators"]
    for aggr in ("mean", "sum", "max"):
        ops[f"aggregate_{aggr}"] = O.aggregate(x, ei, aggr).tolist()
    ops["global_mean_pool"] = O.global_mean_pool(x, batch).tolist()
    ops["scatter_mean_row"] = O.scatter_mean(x[ei[1]], ei[0], 5).tolist()
    score, sbatch, sei = sag_kat()
    perm = O.topk(score, 0.5, sbatch)
    fei, _ = O.filter_adj(sei, None, perm, 8)
    ops["sag_topk_perm"] = perm.tolist()
    ops["sag_filter_adj"] = fei.tolist()
    # training step: loss and gradient norms of one step (dropout off), plus BN buffers after it
    cfg = model_cfg(num_layers=3, dropout_rate=0.0)
    m = seeded_model(cfg, reference=True).train()
    b = make_batch(num_graphs=3, nx=7, ny=6)
    y = torch.tensor([0.5, -0.25, 1.0])
    pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
    loss = torch.nn.functional.mse_loss(pred, y)
    loss.backward()
    out["training"]["sage_mean_3x512_step"] = {
        "cfg": cfg, "batch": dict(num_graphs=3, nx=7, ny=6), "y": y.tolist(), "loss": float(loss),
        "pred": pred.detach().double().tolist(),
        "grad_norms": {k: float(p.grad.double().norm()) for k, p in m.named_parameters() if p.grad is not None},
        "no_grad": sorted(k for k, p in m.named_parameters() if p.grad is None),
        "bn0_running_mean_sum": float(m.batch_norms[0].running_mean.double().sum()),
        "bn0_running_var_sum": float(m.batch_norms[0].running_var.double().sum())}
    path = os.path.join(HERE, "oracle_golden.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
