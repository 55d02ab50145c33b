"""Node-level heads (static_disp, static_stress, mode_shape) of hidden_channels = 128 models: the native 128-wide path
(`model.native128_node_head = True`: bg_node_head128 in eval, bg_sgemm in training) against the zero-padded 512-wide
twin, timed alternately in one process.

    python tools/bench_node_head128.py [--steps 20] [--rounds 3] [--warmup 3] [--out FILE.jsonl]

Workloads (6 layers, `mean` pooling):
  eval   configs[1] (256 plates): GraphSage_meanAggr static_disp (out 6) fp16, GraphSage_addAggr_Shared static_stress tf32
  eval   configs[2] (128 stiffened plates): EA_GNN mode_shape fp16
  train  configs[3] batch (16 plates): GraphSage_meanAggr static_stress tf32 and bf16;
         16 stiffened plates (`config_batch(2, num_graphs=16)`): EA_GNN static_stress tf32
An eval step is one forward; a training step is zero_grad -> forward -> MSE against fixed targets -> backward -> Adam.
Both variants start from the same weights; each round times `--steps` steps of one then the other (CUDA events), the
reported ms/step is the median over rounds.  The engine.TIMERS spans of one more pass per variant (a separate,
instrumented run) show where the time goes; for the native eval forward the `node_head` span (bg_node_head128 alone)
is also given as bytes/s: rows read (n x 128 x element size) plus predictions written (n x out x 4), over the span
time, against the 7.7 TB/s of NVIDIA's HGX B200 data sheet.  Before timing, one step of each gives the largest
relative difference between their predictions (and, in training, between their gradients, per parameter,
norm-relative).  One JSON line per workload, with the GPU name and power limit read in the same process."""
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

HBM_PEAK_BYTES_PER_S = 7.7e12            # HGX B200 data sheet, one GPU
ELEM = {"fp16": 2, "bf16": 2, "tf32": 4, "fp32": 4}

# (mode, batch, model_name, prediction_type, use_z_coord, use_rotations, precision)
WORKLOADS = [
    ("eval", "cfg1", "GraphSage_meanAggr", "static_disp", True, True, "fp16"),
    ("eval", "cfg1", "GraphSage_addAggr_Shared", "static_stress", False, False, "tf32"),
    ("eval", "cfg2", "EA_GNN", "mode_shape", False, False, "fp16"),
    ("train", "cfg3", "GraphSage_meanAggr", "static_stress", False, False, "tf32"),
    ("train", "cfg3", "GraphSage_meanAggr", "static_stress", False, False, "bf16"),
    ("train", "cfg2x16", "EA_GNN", "static_stress", False, False, "tf32"),
]


def _batch(kind):
    return {"cfg1": lambda: config_batch(1), "cfg2": lambda: config_batch(2), "cfg3": lambda: config_batch(3),
            "cfg2x16": lambda: config_batch(2, num_graphs=16)}[kind]()


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


def run(mode, kind, name, ptype, z, rot, prec, args, dev, info):
    b = _batch(kind).to(dev)
    torch.manual_seed(0)
    prec_kw = dict(precision=prec) if mode == "eval" else dict(train_precision=prec)
    base = BuckGNN(16, 5, 128, 6, "mean", ptype, use_z_coord=z, use_rotations=rot, model_name=name, dropout_rate=0.1,
                   **prec_kw).to(dev)
    base.train(mode == "train")
    variants = {}
    for label, flag in (("native", True), ("twin", False)):
        m = copy.deepcopy(base)
        m.native128_node_head = flag
        if not flag:
            m._wide = WideTwin(m, m._ctor_kwargs)       # built up front: its initialisation draws from torch's generator
        variants[label] = (m, torch.optim.Adam(m.parameters(), lr=1e-3) if mode == "train" else None)
    out_dim = base.output_dim
    target = torch.randn(b.num_nodes, out_dim, generator=torch.Generator().manual_seed(3)).to(dev) + 1.0

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
    preds, grads = {}, {}
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
    pred_diff = _rel(preds["native"], preds["twin"])
    grad_diff = max(_rel(grads["native"][k], grads["twin"][k]) for k in grads["twin"]) if grads else None

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
    spans, head_calls = {}, {}
    for label in variants:                              # instrumented pass: spans per step
        engine.TIMERS.enable()
        for _ in range(args.steps):
            step(label)
        summ = engine.TIMERS.summary()
        spans[label] = {k: round(v[0] / args.steps, 4) for k, v in summ.items()}
        head_calls[label] = summ.get("node_head", (0.0, 0))
        engine.TIMERS.disable()
    assert variants["native"][0]._wide is None and variants["twin"][0]._wide is not None
    med = {label: statistics.median(v) for label, v in ms.items()}
    line = {
        "config": f"{kind} ({b.num_graphs} graphs), {name} 6x128 {ptype} (out {out_dim}), mean pooling, {mode}"
                  + (", dropout 0.1, Adam, MSE" if mode == "train" else "")
                  + "; native 128-wide vs zero-padded 512-wide twin, timed alternately",
        "mode": mode, "model": name, "prediction_type": ptype, "out_dim": out_dim,
        ("precision" if mode == "eval" else "train_precision"): prec,
        "nodes": b.num_nodes, "edges": b.num_edges, "steps_per_round": args.steps, "rounds": args.rounds,
        "native_ms_per_step": round(med["native"], 4), "twin_ms_per_step": round(med["twin"], 4),
        "speedup": round(med["twin"] / med["native"], 3),
        "native_vs_twin_rel_pred": float(f"{pred_diff:.3e}"),
        "native_ms_rounds": [round(v, 4) for v in ms["native"]], "twin_ms_rounds": [round(v, 4) for v in ms["twin"]],
        "native_spans_ms_per_step": spans["native"], "twin_spans_ms_per_step": spans["twin"], **info}
    if grad_diff is not None:
        line["native_vs_twin_max_rel_grad"] = float(f"{grad_diff:.3e}")
    if mode == "eval":
        total_ms, calls = head_calls["native"]
        per_call_s = total_ms * 1e-3 / max(calls, 1)
        nbytes = b.num_nodes * 128 * ELEM[prec] + b.num_nodes * out_dim * 4
        line.update({"native_node_head_ms": round(per_call_s * 1e3, 4), "native_node_head_bytes": nbytes,
                     "native_node_head_bytes_per_s": float(f"{nbytes / per_call_s:.4e}"),
                     "native_node_head_share_of_hbm_peak": round(nbytes / per_call_s / HBM_PEAK_BYTES_PER_S, 3),
                     "native_node_head_byte_bound_ms": round(nbytes / HBM_PEAK_BYTES_PER_S * 1e3, 4),
                     "twin_node_head_ms": round(head_calls["twin"][0] / max(head_calls["twin"][1], 1), 4)})
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
