"""Training step of a hidden_channels = 128 model: the native 128-wide step (`model.native128_train = True`) against the
zero-padded 512-wide twin, timed alternately in one process on the configs[3] batch (tools/bench_train.py: 16 graphs,
`config_batch(3, num_graphs=16)`), 6 layers, dropout 0.1.

    python tools/bench_train128.py [--steps 20] [--rounds 5] [--warmup 5] [--out FILE.jsonl]

One step = zero_grad -> model(...) in train mode -> relative-error loss -> loss.backward() -> Adam step.  Both variants
start from the same weights; each round times `--steps` steps of one then the other (CUDA events), and the reported
ms/step is the median over rounds.  The engine.TIMERS spans of one more pass per variant (a separate, instrumented
run) show where the time goes.  One JSON line per (model, train_precision), with the GPU name and power limit read in
the same process."""
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
from buckgnn_b200.synth import config_batch
from tools.bench_narrow import gpu_info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--models", default="GraphSage_addAggr_Shared,GraphSage_meanAggr")
    ap.add_argument("--precisions", default="tf32,bf16")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    capi.device_check()
    info = gpu_info(dev)
    b = config_batch(3, num_graphs=args.graphs).to(dev)
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
                m.native128_train = flag
                variants[label] = (m, torch.optim.Adam(m.parameters(), lr=1e-3))

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
                "config": f"cfg3 batch ({args.graphs} graphs), {name} 6x128, dropout 0.1, Adam; native 128-wide step vs "
                          f"zero-padded 512-wide twin, timed alternately",
                "model": name, "train_precision": prec, "nodes": b.num_nodes, "edges": b.num_edges,
                "steps_per_round": args.steps, "rounds": args.rounds,
                "native_ms_per_step": round(med["native"], 4), "twin_ms_per_step": round(med["twin"], 4),
                "native_graphs_per_s": round(args.graphs / (med["native"] * 1e-3), 1),
                "twin_graphs_per_s": round(args.graphs / (med["twin"] * 1e-3), 1),
                "speedup": round(med["twin"] / med["native"], 3),
                "native_ms_rounds": [round(v, 4) for v in ms["native"]], "twin_ms_rounds": [round(v, 4) for v in ms["twin"]],
                "native_spans_ms_per_step": spans["native"], "twin_spans_ms_per_step": spans["twin"], **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
