"""Training step of a hidden_channels = 128 EA-GNN model: the native 128-wide step (`model.native128_eagnn_train = True`)
against the zero-padded 512-wide twin, timed alternately in one process on 16 stiffened plates
(`config_batch(2, num_graphs=16)`, as tools/bench_train.py --model EA_GNN), 6 layers, `mean` pooling, dropout 0.1.

    python tools/bench_eagnn_train128.py [--steps 10] [--rounds 5] [--warmup 3] [--out FILE.jsonl]

One step = zero_grad -> model(...) in train mode -> EigenvalueRelativeLoss -> loss.backward() -> Adam step.  Both variants
start from the same weights; each round times `--steps` steps of one then the other (CUDA events), and the reported
ms/step is the median over rounds.  The engine.TIMERS spans of one more pass per variant (a separate, instrumented run)
show where the time goes.  Before timing, one step of each from the same weights and the same dropout seed gives the
largest relative difference between their predictions and between their gradients (per parameter, norm-relative).  One
JSON line per (model, train_precision), with the GPU name and power limit read in the same process."""
import argparse
import copy
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from buckgnn_b200 import capi, engine
from buckgnn_b200.loss import EigenvalueRelativeLoss
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import config_batch
from tools.bench_narrow import gpu_info


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=16)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--models", default="EA_GNN,EA_GNN_Shared")
    ap.add_argument("--precisions", default="tf32,bf16")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    capi.device_check()
    info = gpu_info(dev)
    b = config_batch(2, num_graphs=args.graphs).to(dev)
    y = b.y.to(dev).abs() + 0.5
    crit = EigenvalueRelativeLoss(scale=1.0, center=0.0)
    lines = []
    for name in args.models.split(","):
        for prec in args.precisions.split(","):
            torch.manual_seed(0)
            base = BuckGNN(16, 5, 128, 6, "mean", model_name=name, dropout_rate=0.1, train_precision=prec).to(dev).train()
            variants = {}
            for label, flag in (("native", True), ("twin", False)):
                m = copy.deepcopy(base)
                m.native128_eagnn_train = flag
                if not flag:
                    m._wide = WideTwin(m, m._ctor_kwargs)       # built up front: its initialisation draws from torch's generator
                variants[label] = (m, torch.optim.Adam(m.parameters(), lr=1e-3))

            # native against twin after one step from the same weights and the same dropout seed draw
            preds, grads = {}, {}
            for label, (m, _) in variants.items():
                torch.manual_seed(7)
                m.zero_grad(set_to_none=True)
                pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
                crit(pred, y).backward()
                preds[label] = pred.detach().float()
                grads[label] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
            assert grads["native"].keys() == grads["twin"].keys()
            pred_diff = ((preds["native"] - preds["twin"]).abs() / preds["twin"].abs().clamp(min=1e-6)).max().item()
            grad_diff = max(_rel(grads["native"][k], grads["twin"][k]) for k in grads["twin"])

            def step(label):
                m, opt = variants[label]
                opt.zero_grad(set_to_none=True)
                pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
                loss = crit(pred, y)
                loss.backward()
                opt.step()
                return loss

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
                "config": f"cfg2 stiffened plates ({args.graphs} graphs), {name} 6x128, mean pooling, dropout 0.1, Adam, "
                          f"EigenvalueRelativeLoss; native 128-wide step vs zero-padded 512-wide twin, timed alternately",
                "model": name, "train_precision": prec, "nodes": b.num_nodes, "edges": b.num_edges,
                "steps_per_round": args.steps, "rounds": args.rounds,
                "native_ms_per_step": round(med["native"], 4), "twin_ms_per_step": round(med["twin"], 4),
                "native_graphs_per_s": round(args.graphs / (med["native"] * 1e-3), 1),
                "twin_graphs_per_s": round(args.graphs / (med["twin"] * 1e-3), 1),
                "speedup": round(med["twin"] / med["native"], 3),
                "native_vs_twin_max_rel_pred": float(f"{pred_diff:.3e}"),
                "native_vs_twin_max_rel_grad": float(f"{grad_diff:.3e}"),
                "native_ms_rounds": [round(v, 4) for v in ms["native"]], "twin_ms_rounds": [round(v, 4) for v in ms["twin"]],
                "native_spans_ms_per_step": spans["native"], "twin_spans_ms_per_step": spans["twin"], **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
            del variants, base
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
