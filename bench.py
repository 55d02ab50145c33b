#!/usr/bin/env python
"""bench.py -- graphs/sec of the BuckGNN 6x512 GraphSAGE forward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one `model(x, edge_index, edge_attr, batch)` call on one synthetic batch
of BASELINE.json configs[1] (256 non-stiffened plate meshes, super node + hub edges,
random-init weights), CSR build included.  N > 1 (torchrun): every rank runs its own
256 graphs (graph-sharded inference, no collective on the data path; weak scaling).
Prints ONE JSON line (rank 0).

Inputs and weights are generated from fixed seeds, so two runs with the same arguments see
the same data.  `--dump-outputs DIR` writes what the last timed step returned, `(pred, batch)`
of rank 0, as DIR/pred.npy and DIR/batch.npy, so that two builds can be compared output
for output.  With mean pooling `batch` is the input batch vector handed back unchanged, so
pred.npy carries everything the step computed.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "BuckGNN GraphSage_meanAggr 6x512 inference, batch 256 synthetic non-stiffened plate meshes " \
           "(super node + hub edges), BASELINE.json configs[1]"
MODEL_CFG = dict(num_node_features=16, num_edge_features=5, hidden_channels=512, num_layers=6,
                 pooling_layer="mean", model_name="GraphSage_meanAggr")
GRAPHS_PER_RANK = 256
CPU_SAMPLE_GRAPHS = 16


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def _traffic_from_profile(name_part: str, exclude: str = ""):
    """Measured DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the kernel whose name
    contains `name_part`, averaged over the launches of the newest committed `ncu --set full` summary
    (profiles/r*_ncu_full_summary.csv, written by tools/ncu_summary.py).  None if there is no capture."""
    import csv
    import glob
    import re

    def version(path):                      # profiles/rNN_vMM_ncu_full_summary.csv -> (NN, MM)
        m = re.search(r"r(\d+)_v(\d+)_ncu_full_summary", os.path.basename(path))
        return (int(m.group(1)), int(m.group(2))) if m else (-1, -1)
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_summary.csv")), key=version)
    if not files:
        return None
    rows = list(csv.reader(open(files[-1])))
    if len(rows) < 3:
        return None
    hdr, units = rows[0], rows[1]
    try:
        i_n, i_r, i_w = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    except ValueError:
        return None
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    vals = [float(r[i_r]) * scale.get(units[i_r], 1.0) + float(r[i_w]) * scale.get(units[i_w], 1.0)
            for r in rows[2:] if name_part in r[i_n] and not (exclude and exclude in r[i_n])]
    return {"bytes_per_launch": sum(vals) / len(vals), "launches": len(vals),
            "source": os.path.relpath(files[-1], ROOT)} if vals else None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every tensor as out_dir/<name>.npy: floating point as float32 (float64 stays float64), integers as
    float64, which holds them exactly.  The files stay within DUMP_BYTES in all: an array larger than its share is
    replaced by a sample of its rows, drawn with a fixed seed so that every run keeps the same rows."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach().cpu()
        a = (t.float() if t.is_floating_point() and t.dtype != torch.float64 else t.double()).numpy()
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons.  Started BEFORE the warm-up (nvidia-smi takes a while to
    come up); `begin()` / `end()` bracket the timed region and only samples that arrived inside it are summarised
    (if the region was shorter than the sampling period, the sample nearest to it is used and flagged)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def wait_ready(self, timeout: float = 5.0):
        t = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        rows = self.rows
        inside = [r for t, r in rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t)]
        how = "inside the timed region"
        if not inside and rows and self.t0 is not None:
            mid = 0.5 * (self.t0 + (self.t1 or self.t0))
            inside = [min(rows, key=lambda tr: abs(tr[0] - mid))[1]]
            how = "nearest sample (timed region shorter than the sampling period)"
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "sampled": how}


def _oracle_model():
    import torch
    from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats
    torch.manual_seed(0)
    ref = OracleBuckGNN(**MODEL_CFG).eval()
    randomize_bn_stats(ref, realistic=True)
    return ref


def cpu_oracle_throughput(steps: int, warmup: int):
    """The pure-torch CPU restatement of the reference forward on a bounded sample."""
    import torch
    from buckgnn_b200.synth import config_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _oracle_model()
    b = config_batch(1, num_graphs=CPU_SAMPLE_GRAPHS)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            outs = ref(b.x, b.edge_index, b.edge_attr, b.batch)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return dict(value=CPU_SAMPLE_GRAPHS / t, unit="graphs/s", cores=cores, kind="port",
                sample=f"first {CPU_SAMPLE_GRAPHS} graphs of the workload ({b.num_nodes} nodes, {b.num_edges} edges), "
                       f"{steps} timed forwards after {warmup} warm-up, torch fp32 oracle"), t, outs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    cpu, t, outs = cpu_oracle_throughput(steps, warmup)
    line = {"metric": "graphs/sec", "value": cpu["value"], "unit": "graphs/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "sample": cpu["sample"]},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "PyG/torch_scatter are not installable here; this is the CPU oracle port of the reference forward"}
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("pred", "batch"), outs)))


def modes_section(args, dev, resident, world, G, barrier):
    """The other operand modes on the same workload (north_star: rtol 1e-4 in an fp32-GEMM mode): graphs/s over a few steps."""
    import torch
    import torch.distributed as dist
    from buckgnn_b200.model import BuckGNN
    ref = _oracle_model()
    out = {}
    for mode in ("tf32", "fp32"):
        m = BuckGNN(**MODEL_CFG, precision=mode, cta_group=args.cta_group)
        m.load_state_dict(ref.state_dict())
        m = m.to(dev).eval()
        with torch.no_grad():
            for _ in range(2):
                m(resident.x, resident.edge_index, resident.edge_attr, resident.batch)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = max(2, min(args.steps, 5))
            e0.record()
            for _ in range(n):
                m(resident.x, resident.edge_index, resident.edge_attr, resident.batch)
            e1.record()
            barrier()
        ms = e0.elapsed_time(e1) / n
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        out[mode] = {"graphs_per_s": world * G / (ms * 1e-3), "ms_per_step": ms, "steps": n,
                     "what": "fp32 storage, tf32 operands" if mode == "tf32" else "fp32-GEMM mode (3xTF32 split operands)"}
        del m
    # the fused SAGE layer (bg_sage_fused512: aggregate operand gathered inside the update GEMM), headline precision
    m = BuckGNN(**MODEL_CFG, precision=args.precision, cta_group=args.cta_group)
    m.load_state_dict(ref.state_dict())
    m = m.to(dev).eval()
    if __import__("buckgnn_b200.engine", fromlist=["x"]).can_fuse_aggregate(m.precision, "mean", True):
        with torch.no_grad():
            plain, _ = m(resident.x, resident.edge_index, resident.edge_attr, resident.batch)
            m.fuse_aggregate = True
            fused, _ = m(resident.x, resident.edge_index, resident.edge_attr, resident.batch)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 2
            e0.record()
            for _ in range(n):
                m(resident.x, resident.edge_index, resident.edge_attr, resident.batch)
            e1.record()
            barrier()
        ms = e0.elapsed_time(e1) / n
        dev_rel = ((fused.float() - plain.float()).abs() / plain.float().abs().clamp(min=1e-3)).max().item()
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        out["fused_sage_layer"] = {"graphs_per_s": world * G / (ms * 1e-3), "ms_per_step": ms, "steps": n,
                                   "max_rel_dev_from_default_path": dev_rel,
                                   "what": "opt-in: every SAGE layer as one kernel, the aggregate never written to HBM "
                                           "(bit-identical operand; slower: gather-latency-bound, DESIGN.md section 5)"}
    del m
    return out


def train_section(args, dev, world, rank, barrier):
    """BASELINE.json configs[3]: TRAIN_FINAL-style training step, GraphSage_meanAggr 6x512, 16 graphs per GPU, dropout
    0.1, relative-error loss, Adam; graph-sharded, gradients all-reduced (mean) over NCCL from one flat buffer
    (dist.GradSync: buckets of >= 8 M elements can start under the backward pass; this model's 3.3 M go in one collective).  `allreduce_exposed_ms` = step time with the collectives - step time without them."""
    import torch
    import torch.distributed as dist
    from buckgnn_b200.loss import EigenvalueRelativeLoss
    from buckgnn_b200.model import BuckGNN
    from buckgnn_b200.synth import config_batch
    torch.manual_seed(0)                                    # same initial weights on every rank
    cfg = dict(MODEL_CFG, dropout_rate=0.1)
    model = BuckGNN(**cfg, train_precision=args.train_precision).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    b = config_batch(3, rank=rank, num_graphs=16).to(dev)
    y = b.y.abs() + 0.5
    crit = EigenvalueRelativeLoss(scale=1.0, center=0.0)
    sync = model.enable_gradient_sync() if world > 1 else None
    steps = max(3, min(args.steps, 20))

    def step():
        opt.zero_grad(set_to_none=True)
        pred, _ = model(b.x, b.edge_index, b.edge_attr, b.batch)
        loss = crit(pred, y)
        loss.backward()
        opt.step()
        return loss

    def timed(n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            last = step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / n
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, float(last.detach())

    for _ in range(3):
        first = step()
    ms, loss_last = timed(steps)
    out = {"config": f"BASELINE.json configs[3]: training step GraphSage_meanAggr 6x512, 16 graphs per GPU, dropout 0.1, Adam, "
                     f"graph-sharded x{world}", "train_precision": args.train_precision, "ms_per_step": ms, "steps": steps,
           "graphs_per_s": world * 16 / (ms * 1e-3), "nodes_per_gpu": b.num_nodes, "loss_first": float(first.detach()),
           "loss_last": loss_last}
    if sync is not None:
        sync.time_collectives = True                        # one instrumented step: device time of every collective
        step()
        torch.cuda.synchronize()
        out["allreduce_ms"] = sum(a.elapsed_time(c) for a, c in sync.events)
        out["allreduce_buckets"] = len(sync.events)
        out["allreduce_elements"] = int(sync.flat.numel())
        sync.time_collectives = False
        model._grad_sync = None                             # the same steps without any collective (ranks diverge: timing only)
        step()
        ms_local, _ = timed(steps)
        out["ms_per_step_without_allreduce"] = ms_local
        out["allreduce_exposed_ms"] = ms - ms_local
        out["allreduce"] = ("one flat fp32 gradient buffer the backward kernels write into; ncclAllReduce(avg) on a second stream in "
                            "buckets of >= 8 M elements (latency-bound collectives: one for this model; dist.GradSync)")
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from buckgnn_b200 import capi, engine
    from buckgnn_b200.model import BuckGNN
    from buckgnn_b200.synth import config_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    capi.device_check()
    peaks = _peaks()

    # ---- model: same seeded weights as the oracle, default precision
    ref = _oracle_model()
    model = BuckGNN(**MODEL_CFG, precision=args.precision, cta_group=args.cta_group)
    model.load_state_dict(ref.state_dict())
    model = model.to(dev).eval()

    # ---- workload: this rank's shard of graphs, pinned on the host
    host = config_batch(1, rank=rank, num_graphs=args.graphs).pin_memory()
    G, N, E = host.num_graphs, host.num_nodes, host.num_edges
    resident = host.to(dev)
    def forward(b):
        with torch.no_grad():
            return model(b.x, b.edge_index, b.edge_attr, b.batch)

    def fwd(b):
        return forward(b)[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity check of this very configuration on a sample (not timed)
    sample = config_batch(1, rank=rank, num_graphs=4)
    with torch.no_grad():
        want = ref(sample.x, sample.edge_index, sample.edge_attr, sample.batch)[0]
    got = fwd(sample.to(dev)).cpu()
    rel_err = ((got - want).abs() / want.abs().clamp(min=1e-3)).max().item()

    # ---- device-resident timing (the `value`)
    with ClockSampler(local) as clk:
        for _ in range(args.warmup):
            fwd(resident)
        clk.wait_ready()
        barrier()
        engine.TIMERS.enable()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clk.begin()
        ev0.record()
        for _ in range(args.steps):
            outs = forward(resident)
        ev1.record()
        barrier()
        clk.end()
    step_ms = ev0.elapsed_time(ev1) / args.steps
    # (pred, batch) of the last timed step, on the host before any later forward runs
    last_outs = dict(zip(("pred", "batch"), (t.cpu() for t in outs))) if args.dump_outputs else None
    kernel_ms = engine.TIMERS.summary()          # per kernel class: total ms, calls
    engine.TIMERS.disable()

    # second figure (SURVEY.md section 8d): the same steps with the CSR cache warm -- `cache_index=True` keeps the
    # index of an unchanged `edge_index` tensor, as a serving loop over a fixed mesh set would
    model.cache_index = True
    for _ in range(2):
        fwd(resident)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(args.steps):
        fwd(resident)
    c1.record()
    barrier()
    cached_ms = c0.elapsed_time(c1) / args.steps
    model.cache_index = False
    model._index_cache = None

    # ---- end to end: every step copies that step's pinned-host inputs H->D (x, edge_index, edge_attr,
    # batch, y, ptr: everything `batch.to(device)` moves) and reads pred back D->H.  The copies of
    # step i+1 run on a second stream while step i computes, and the result of step i reaches the host while
    # step i+1 computes (buckgnn_b200.pipeline.PipelinedInference); every result is on the host inside the clock.
    from buckgnn_b200.pipeline import PipelinedInference, WireBatch
    h2d_full = sum(t.numel() * t.element_size() for t in (host.x, host.edge_index, host.edge_attr, host.batch,
                                                           host.y, host.ptr))
    # GraphSAGE never reads edge_attr / y / ptr, and the super node's hub pairs (1/3 of edge_index) follow from the node
    # offsets: the loader hands the pipeline the compact wire format (x, explicit edges as int32, three offset vectors)
    # and bg_expand_wire rebuilds the exact PyG tensors on the device (tests/test_gpu_kernels.py)
    wire = WireBatch.from_batch(host).pin_memory()
    h2d = wire.nbytes()
    copy_ms, fwd_dev_ms, stamps = [], [], []
    # the loop object is created once (as an inference service would): its two device-side staging batches and its
    # pinned result buffers are set up by the warm-up pass, not inside the timed region
    pipe = PipelinedInference(model, (), dev, depth=1)
    pipe.prefetcher.time_copies = True

    def e2e_run(n):
        outs = None
        evs = {}

        def hook(step, before):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            evs.setdefault(step, []).append(ev)
        pipe.on_launch = hook
        pipe.prefetcher.copy_events = []
        seen = 0
        stamps[:] = [time.perf_counter()]
        for step, pred_host in pipe.run(wire for _ in range(n)):   # pred_host: this step's eigenvalues, on the host
            outs = pred_host
            seen += 1
            stamps.append(time.perf_counter())
        assert seen == n
        torch.cuda.synchronize()
        copy_ms[:] = [a.elapsed_time(b_) for a, b_ in pipe.prefetcher.copy_events]
        fwd_dev_ms[:] = [a.elapsed_time(b_) for a, b_ in evs.values()]
        return outs
    e2e_run(max(2, args.warmup // 2))
    barrier()
    t0 = time.perf_counter()
    out = e2e_run(args.steps)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps    # host wall clock: includes every copy and sync
    barrier()
    # diagnostic: same loop without the H2D copies (resident batch, pred.cpu() every step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fwd(resident).cpu()
    sync_only_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    barrier()

    # diagnostic (row f1): the dataset lives in HBM, every step collates its batch on the device -- no PCIe traffic
    from buckgnn_b200.collate import DeviceGraphStore
    from buckgnn_b200.synth import make_plate_graph
    store = DeviceGraphStore([make_plate_graph(rank * GRAPHS_PER_RANK + i) for i in range(G)], dev)
    sel = torch.arange(G, device=dev)
    for _ in range(2):
        fwd(store.batch(sel)).cpu()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fwd(store.batch(sel)).cpu()
    resident_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    del store
    barrier()

    modes = None if args.no_extras else modes_section(args, dev, resident, world, G, barrier)
    del resident
    torch.cuda.empty_cache()
    train_info = None if args.no_extras else train_section(args, dev, world, rank, barrier)

    # ---- max over ranks
    if world > 1:
        t = torch.tensor([step_ms, e2e_ms, cached_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms, e2e_ms, cached_ms = t.tolist()
    value = world * G / (step_ms * 1e-3)
    e2e_value = world * G / (e2e_ms * 1e-3)

    if rank == 0:
        esz = 4 if args.precision in ("tf32", "fp32") else 2
        L = MODEL_CFG["num_layers"]
        # algorithmic work per launch (DESIGN.md section 5)
        agg_bytes = 2 * N * 512 * esz + 4 * E + 4 * (N + 1)
        upd_flops = 2.0 * N * 1024 * 512 * (3 if args.precision == "fp32" else 1)    # layers 1..L-1 (layer 0 is folded: K = 320)
        tf_peak = peaks["tf_sustained"] * (0.5 if esz == 4 else 1.0)
        roofs = {}
        if "aggregate" in kernel_ms:
            ms, calls = kernel_ms["aggregate"]
            a = agg_bytes / (ms / calls * 1e-3) / 1e9
            tr = _traffic_from_profile("k_aggregate_rows<", exclude="rows128") if args.precision == "fp16" else None
            roofs["aggregate"] = {"bound": "hbm", "achieved": a, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                  "frac": a / peaks["hbm_gbs"], "traffic": tr and tr["bytes_per_launch"],
                                  "traffic_source": tr and tr["source"], "algorithmic_bytes": agg_bytes,
                                  "kernel": "k_aggregate_rows (hub-streaming warps) + k_hub_finalize",
                                  "ms_per_launch": ms / calls, "share_of_step": ms / args.steps / step_ms}
        fused_pool = "sage_update_pool" in kernel_ms      # last layer: rows summed for the pooling layer, not stored
        if "sage_update" in kernel_ms:
            ms, calls = kernel_ms["sage_update"]
            if fused_pool:                               # same kernel, pool-fused epilogue instance: same flops
                ms, calls = ms + kernel_ms["sage_update_pool"][0], calls + kernel_ms["sage_update_pool"][1]
            a = upd_flops / (ms / calls * 1e-3) / 1e12
            tr = _traffic_from_profile("k_gemm512<2, __half, 1,") if args.precision == "fp16" else None
            roofs["sage_update"] = {"bound": "tensor", "achieved": a, "peak": tf_peak, "unit": "TFLOP/s",
                                    "frac": a / tf_peak, "traffic": tr and tr["bytes_per_launch"],
                                    "traffic_source": tr and tr["source"], "algorithmic_flops": upd_flops,
                                    "kernel": "k_gemm512" + (" (incl. the pool-fused last layer)" if fused_pool else ""),
                                    "ms_per_launch": ms / calls, "share_of_step": ms / args.steps / step_ms}
        dominant = max(roofs, key=lambda k: roofs[k]["share_of_step"]) if roofs else None
        # whole-step fraction (SURVEY.md section 8d): sum over the kernel classes of max(bytes / HBM peak, flops / tensor
        # peak) divided by the measured step -- algorithmic work only (DESIGN.md section 5)
        ideal = {
            "csr_build": (16.0 * E + 8.0 * E + 8.0 * N) / peaks["hbm_gbs"] / 1e6,
            "encoder_front": (N * 16 * 4 + N * 128 * esz) / peaks["hbm_gbs"] / 1e6,
            "aggregate128": (2 * N * 128 * esz + 4 * E + 4 * (N + 1)) / peaks["hbm_gbs"] / 1e6,
            "sage_update0": max(2.0 * N * 320 * 512 * (3 if args.precision == "fp32" else 1) / tf_peak / 1e9,
                                (N * (320 + 512) * esz) / peaks["hbm_gbs"] / 1e6),
            "aggregate": (L - 1) * agg_bytes / peaks["hbm_gbs"] / 1e6,
            "sage_update": (L - 1 - int(fused_pool)) * max(upd_flops / tf_peak / 1e9, N * (1024 + 512 + 512) * esz / peaks["hbm_gbs"] / 1e6),
            "pool_head": N * 512 * esz / peaks["hbm_gbs"] / 1e6,
        }
        if fused_pool:      # the last layer writes [N/32, 512] f32 block sums instead of [N, 512] rows; the pool reads those
            ideal["sage_update_pool"] = max(upd_flops / tf_peak / 1e9, (N * 1024 * esz + N / 32 * 512 * 4) / peaks["hbm_gbs"] / 1e6)
            ideal["pool_head"] = (N / 32 * 512 * 4) / peaks["hbm_gbs"] / 1e6
        step_roofline = {"ideal_ms": sum(ideal.values()), "measured_ms": step_ms, "frac": sum(ideal.values()) / step_ms,
                         "ideal_ms_by_kernel": ideal,
                         "note": "sum_k max(B_k / measured HBM peak, F_k / measured sustained tensor peak) / step time"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu, _, _ = cpu_oracle_throughput(3, 1)
        line = {
            "metric": "graphs/sec", "value": value, "unit": "graphs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"fp16": "f16", "bf16": "bf16", "tf32": "tf32",
                                           "fp32": "f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "graphs_per_gpu": G, "nodes_per_gpu": N, "edges_per_gpu": E,
                       "precision": args.precision, "cta_group": args.cta_group, "csr_build": "inside timed region",
                       "layer0": "encoder Linear(128,512) folded into SAGE layer 0 (exact algebra)",
                       "last_layer": ("epilogue sums its rows per 32-row block for global_mean_pool instead of storing them "
                                      "(pool-fused)") if fused_pool else "rows stored, pooled by bg_pool_head",
                       "l2": "inputs+activations (>2 GB per step) exceed the 126 MB L2; no explicit flush",
                       "parallelism": f"graph-sharded x{world}, no data-path collective",
                       "parity_rel_err_vs_oracle_sample": rel_err},
            "e2e": {"value": e2e_value, "unit": "graphs/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "h2d_bytes_full_pyg_batch": h2d_full,
                    "wire_format": "x f32 + explicit edges int32 + node/edge offsets; hub pairs, batch vector and int64 "
                                   "widening rebuilt on the device (bg_expand_wire); edge_attr / y / ptr are never read by "
                                   "GraphSAGE and stay on the host",
                    "d2h_bytes_per_step": int(out.numel() * out.element_size()),
                    "ms_per_step_without_h2d": sync_only_ms,
                    "ms_per_step_device_collate": resident_ms,      # DeviceGraphStore.batch() + forward + pred.cpu()
                    "h2d_copy_ms_overlapped": sorted(copy_ms)[len(copy_ms) // 2] if copy_ms else None,
                    "forward_device_ms_under_copy": sorted(fwd_dev_ms)[len(fwd_dev_ms) // 2] if fwd_dev_ms else None,
                    "result_arrival_intervals_ms": [round((b_ - a_) * 1e3, 3) for a_, b_ in zip(stamps, stamps[1:])],
                    "how": "buckgnn_b200.pipeline.PipelinedInference: pinned host batch (wire format) -> H2D of step i+1 on a copy stream "
                           "during step i -> model(...) -> eigenvalues of every step read back to pinned host memory "
                           "(one step late, so the GPU never waits for the host); host wall clock over the timed "
                           "steps, all K results on the host before the clock stops"},
            "gpu_launches": engine.LAUNCHES_PER_FORWARD(L, folded=model.fold_encoder, fused_pool=fused_pool) * args.steps,
            "roofline": roofs.get(dominant),
            "roofline_all": roofs,
            "roofline_step": step_roofline,
            "csr_cache_warm": {"value": world * G / (cached_ms * 1e-3), "unit": "graphs/s", "ms_per_step": cached_ms,
                               "how": "cache_index=True: the CSR of an unchanged edge_index tensor is reused"},
            "kernel_ms_per_step": {k: v[0] / args.steps for k, v in kernel_ms.items()},
            "modes": modes,
            "train": train_info,
            "peaks": peaks,
            "cpu_baseline": cpu,
            "clocks": clk.summary(),
        }
        print(json.dumps(line))
        if last_outs is not None:
            dump_outputs(args.dump_outputs, last_outs)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--cta-group", type=int, default=2)
    ap.add_argument("--graphs", type=int, default=GRAPHS_PER_RANK)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the tf32 / fp32 modes and the training-step section")
    ap.add_argument("--train-precision", default="tf32")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write (pred, batch) of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
