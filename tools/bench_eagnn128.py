"""hidden_channels = 128 EA-GNN inference on the 128-wide kernels (`native128_eagnn`) against the zero-padded 512-wide
twin, in one process.

Workload: BASELINE.json configs[2] as bench.py builds it (128 stiffened plates from `synth`, super node + hub edges,
same generator and seed), 6 layers, `mean` pooling, at hidden 128: EA_GNN in fp16 and in bf16 (the precision BASELINE
names for configs[2]) and EA_GNN_Shared in fp16.  Per case the native path and `narrow.WideTwin` are timed alternately
(CUDA events, after warm-up), then one extra pass per path records the per-kernel spans of engine.TIMERS.  The oracle
comparison runs on a 16-graph sample of the same generator.  One JSON line per case:

    python tools/bench_eagnn128.py [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [("EA_GNN", "fp16"), ("EA_GNN", "bf16"), ("EA_GNN_Shared", "fp16")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations native / twin")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_eagnn128.jsonl"))
    args = ap.parse_args()

    import torch
    from buckgnn_b200 import capi, engine
    from buckgnn_b200.model import BuckGNN
    from buckgnn_b200.narrow import WideTwin
    from buckgnn_b200.synth import config_batch
    from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats
    from tools.bench_narrow import gpu_info, rel

    capi.device_check()
    dev = torch.device("cuda", 0)
    info = gpu_info(dev)
    batch = config_batch(2).to(dev)
    sample = config_batch(2, num_graphs=16)
    lines = []
    for name, precision in CASES:
        cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=6, pooling_layer="mean",
                   model_name=name)
        torch.manual_seed(0)
        ref = OracleBuckGNN(**cfg).eval()
        randomize_bn_stats(ref, realistic=True)
        model = BuckGNN(**cfg, precision=precision)
        model.load_state_dict(ref.state_dict())
        model.native128_eagnn = True
        model = model.to(dev).eval()
        twin = WideTwin(model, model._ctor_kwargs)
        paths = {"native": lambda b: model(b.x, b.edge_index, b.edge_attr, b.batch)[0],
                 "twin": lambda b: twin.forward(b.x, b.edge_index, b.edge_attr, b.batch)[0]}

        with torch.no_grad():
            for fn in paths.values():
                for _ in range(args.warmup):
                    fn(batch)
            torch.cuda.synchronize()
            times = {k: [] for k in paths}
            for _ in range(args.rounds):
                for key, fn in paths.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(args.steps):
                        fn(batch)
                    e1.record()
                    torch.cuda.synchronize()
                    times[key].append(e0.elapsed_time(e1) / args.steps)
            spans = {}
            for key, fn in paths.items():
                engine.TIMERS.enable()
                fn(batch)
                spans[key] = {k: round(ms, 4) for k, (ms, _) in engine.TIMERS.summary().items()}
                engine.TIMERS.disable()
            native = paths["native"](batch).cpu()
            assert model._ran_native128 and model._wide is None      # timed the 128-wide kernels, not the twin
            wide = paths["twin"](batch).cpu()
            want = ref(sample.x, sample.edge_index, sample.edge_attr, sample.batch)[0]
            sd = sample.to(dev)
            err_oracle = {k: rel(fn(sd).cpu(), want) for k, fn in paths.items()}
        G = batch.num_graphs
        res = {"model": name, "precision": model.precision, "hidden_channels": 128, "num_layers": 6, "pooling": "mean",
               "workload": f"BASELINE.json configs[2]: {G} graphs, {batch.num_nodes} nodes, {batch.num_edges} edges",
               **info, "steps": args.steps, "rounds": args.rounds}
        for key in paths:
            best = min(times[key])
            res[key] = {"ms_per_forward": round(best, 4), "ms_per_forward_all_rounds": [round(t, 4) for t in times[key]],
                        "graphs_per_s": round(G / best * 1e3, 1), "kernel_spans_ms": spans[key],
                        "max_rel_err_vs_oracle_16_graphs": err_oracle[key]}
        res["speedup"] = round(min(times["twin"]) / min(times["native"]), 3)
        res["max_rel_diff_native_vs_twin"] = rel(native, wide)
        lines.append(res)
        print(json.dumps(res), flush=True)
        del model, twin, paths
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
