"""SAGPooling variants (GraphSAGE_SAG, EAGNN_SAG) of hidden_channels = 128 models: the native 128-wide path
(`model.native128_sag = True`) against the zero-padded 512-wide twin, timed alternately in one process.

    python tools/bench_sag128.py [--steps 20] [--rounds 3] [--warmup 3] [--out FILE.jsonl]

Workloads (6 layers, `mean` pooling, eigenvalue head):
  eval   configs[1] (256 plates): GraphSAGE_SAG in fp32 (its default: the 3xTF32 fp32-GEMM mode) and in fp16
  eval   configs[2] (128 stiffened plates): EAGNN_SAG in tf32 (its default)
  train  configs[3] batch (16 plates): GraphSAGE_SAG tf32 and bf16;
         16 stiffened plates (`config_batch(2, num_graphs=16)`): EAGNN_SAG tf32
An eval step is one forward; a training step is zero_grad -> forward -> MSE against fixed targets -> backward -> Adam.
Both variants start from the same weights; each round times `--steps` steps of one then the other (CUDA events), the
reported ms/step is the median over rounds.  The engine.TIMERS spans of one more pass per variant (a separate,
instrumented run) show where the time goes.  Before timing, one step of each gives the relative difference between
their predictions, how many of the selected nodes differ (the selection is a discrete function of a rounded score:
threshold nodes may change sides), and in training the largest per-parameter norm-relative gradient difference when
both select the same nodes.  One JSON line per workload, with the GPU name and power limit read in the same process."""
import argparse
import copy
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
from buckgnn_b200 import capi, engine
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import config_batch
from tools.bench_narrow import gpu_info

# (mode, batch, model_name, precision)
WORKLOADS = [
    ("eval", "cfg1", "GraphSAGE_SAG", "fp32"),
    ("eval", "cfg1", "GraphSAGE_SAG", "fp16"),
    ("eval", "cfg2", "EAGNN_SAG", "tf32"),
    ("train", "cfg3", "GraphSAGE_SAG", "tf32"),
    ("train", "cfg3", "GraphSAGE_SAG", "bf16"),
    ("train", "cfg2x16", "EAGNN_SAG", "tf32"),
]


def _batch(kind):
    return {"cfg1": lambda: config_batch(1), "cfg2": lambda: config_batch(2), "cfg3": lambda: config_batch(3),
            "cfg2x16": lambda: config_batch(2, num_graphs=16)}[kind]()


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


def run(mode, kind, name, prec, args, dev, info):
    b = _batch(kind).to(dev)
    torch.manual_seed(0)
    prec_kw = dict(precision=prec) if mode == "eval" else dict(train_precision=prec)
    base = BuckGNN(16, 5, 128, 6, "mean", model_name=name, dropout_rate=0.1, **prec_kw).to(dev)
    base.train(mode == "train")
    variants = {}
    for label, flag in (("native", True), ("twin", False)):
        m = copy.deepcopy(base)
        m.native128_sag = flag
        if not flag:
            m._wide = WideTwin(m, m._ctor_kwargs)       # built up front: its initialisation draws from torch's generator
        variants[label] = (m, torch.optim.Adam(m.parameters(), lr=1e-3) if mode == "train" else None)
    n_graphs = int(b.batch.max()) + 1
    target = torch.randn(n_graphs, generator=torch.Generator().manual_seed(3)).to(dev) + 1.0

    def step(label):
        m, opt = variants[label]
        if mode == "eval":
            with torch.no_grad():
                return m(b.x, b.edge_index, b.edge_attr, b.batch)[0]
        opt.zero_grad(set_to_none=True)
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, target).backward()
        opt.step()
        return pred

    # native against twin from the same weights (and, in training, the same dropout seed draw)
    preds, grads, perms = {}, {}, {}
    for label, (m, _) in variants.items():
        torch.manual_seed(7)
        if mode == "eval":
            with torch.no_grad():
                preds[label] = m(b.x, b.edge_index, b.edge_attr, b.batch)[0].float()
        else:
            m.zero_grad(set_to_none=True)
            pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
            F.mse_loss(pred, target).backward()
            preds[label] = pred.detach().float()
            grads[label] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
        perms[label] = m.last_pool.perm.long().cpu()
    pred_diff = _rel(preds["native"], preds["twin"])
    same_selection = torch.equal(perms["native"], perms["twin"])
    nodes_differ = len(set(perms["native"].tolist()) ^ set(perms["twin"].tolist()))
    grad_diff = (max(_rel(grads["native"][k], grads["twin"][k]) for k in grads["twin"])
                 if grads and same_selection else None)

    for label in variants:
        for _ in range(args.warmup):
            step(label)
    torch.cuda.synchronize()
    ms = {label: [] for label in variants}
    for _ in range(args.rounds):
        for label in variants:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(label)
            e1.record()
            torch.cuda.synchronize()
            ms[label].append(e0.elapsed_time(e1) / args.steps)
    spans = {}
    for label in variants:                              # instrumented pass: spans per step
        engine.TIMERS.enable()
        for _ in range(args.steps):
            step(label)
        spans[label] = {k: round(v[0] / args.steps, 4) for k, v in engine.TIMERS.summary().items()}
        engine.TIMERS.disable()
    assert variants["native"][0]._wide is None and variants["twin"][0]._wide is not None
    med = {label: statistics.median(v) for label, v in ms.items()}
    line = {
        "config": f"{kind} ({n_graphs} graphs), {name} 6x128 buckling, mean pooling, {mode}"
                  + (", dropout 0.1, Adam, MSE" if mode == "train" else "")
                  + "; native 128-wide vs zero-padded 512-wide twin, timed alternately",
        "mode": mode, "model": name, ("precision" if mode == "eval" else "train_precision"): prec,
        "nodes": b.num_nodes, "edges": b.num_edges, "pooled_nodes": int(perms["native"].numel()),
        "steps_per_round": args.steps, "rounds": args.rounds,
        "native_ms_per_step": round(med["native"], 4), "twin_ms_per_step": round(med["twin"], 4),
        "speedup": round(med["twin"] / med["native"], 3),
        "native_vs_twin_rel_pred": float(f"{pred_diff:.3e}"),
        "native_vs_twin_same_selection": same_selection, "native_vs_twin_selected_nodes_differ": nodes_differ,
        "native_ms_rounds": [round(v, 4) for v in ms["native"]], "twin_ms_rounds": [round(v, 4) for v in ms["twin"]],
        "native_spans_ms_per_step": spans["native"], "twin_spans_ms_per_step": spans["twin"], **info}
    if grad_diff is not None:
        line["native_vs_twin_max_rel_grad"] = float(f"{grad_diff:.3e}")
    del variants, base
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default=None, help="comma-separated indices into WORKLOADS")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    capi.device_check()
    info = gpu_info(dev)
    picks = range(len(WORKLOADS)) if args.only is None else [int(i) for i in args.only.split(",")]
    lines = []
    for i in picks:
        line = run(*WORKLOADS[i], args, dev, info)
        lines.append(line)
        print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
